// ngs-cuda-qc — host driver of the CUDA `ngs qc` path.  Mirrors the reference's subcommand
// (src/qc/command.rs): QcArgs (36-102), qc() (109-218), app() (226-421).  Same positional
// arguments and flags, same checks in the same order, same output file; the two hot loops of
// app() (305-316 and 350-397) are replaced by one pass of the CUDA engine per GPU.  `index` builds the
// BAI that `qc` needs (src/index/bam.rs:39-109) in one pass of the engine.
//
// Every run is a FilePlan: each GPU runs a queue of (file, shard) entries through one engine (stream_queue), and cuts at record
// anchors are proven by the run (run_plan).  A BAM without an index is cut between GPUs at record anchors the engine finds
// (ngsq_find_record), each GPU indexes its part (NGSQ_F_INDEX_PART; one GPU indexes the whole file as one part) and the host
// joins the parts (ngsq_join_bai): `index`, and `qc --cuda-build-index`, which writes the missing index (.bai, or .csi with
// --cuda-csi) in the same pass as the results.  `qc` plans its shards from <BAM>.bai, or from <BAM>.csi when there is no .bai
// (the reference needs the .bai).  `qc --cuda-any-order` reads no index and
// takes records in any order (unsorted, queryname-sorted or collated files): one shard, or cuts at record anchors with every
// reference split between the devices.  `qc --cuda-also <BAM>` adds files of the same sample under the same rules: whole files
// queued on each device (ngsq_next_file between them), or with fewer files than devices each file cut between its devices.
// `qc --cuda-by-read-group` also writes the record facets of every @RG read group, tallied in the same pass (NGSQ_F_READ_GROUPS).
//
//   ngs-cuda-qc qc <BAM> <REFERENCE_GENOME> [-n N] [-o DIR] [-p PREFIX] [--only FACET]
//               [--cuda-devices 0,1,..] [--cuda-build-index [--cuda-csi [--cuda-min-shift N]] | --cuda-any-order] [--cuda-gc-seed S]
//               [--cuda-no-crc] [--cuda-chunk-mb M] [--cuda-buffered-io] [--cuda-perf] [--cuda-also <BAM> ..] [--cuda-by-read-group]
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
#include "read_groups.hpp"

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
  bool any_order = false;    // --cuda-any-order: no index is read, the records may come in any order
  std::vector<std::string> also;  // --cuda-also: more files of the sample, checked with src as one (implies any_order)
  bool by_read_group = false;     // --cuda-by-read-group: one more results JSON per @RG read group
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
    reopen(path, direct);
    for (auto& b : buf_) {
      b = (uint8_t*)ngsq_host_alloc(kLead + chunk_ + 4096);
      if (!b) throw std::runtime_error("cannot allocate pinned staging buffers");
    }
  }
  // reads another file through the same pinned buffers (`--cuda-also`)
  void reopen(const std::string& path, bool direct) {
    if (fd_ >= 0) close(fd_);
    fd_ = -1;
    direct_ = false;
#ifdef O_DIRECT
    if (direct) fd_ = open(path.c_str(), O_RDONLY | O_DIRECT);
    direct_ = fd_ >= 0;
#endif
    if (fd_ < 0) fd_ = open(path.c_str(), O_RDONLY);
    if (fd_ < 0) throw std::runtime_error("cannot open " + path);
  }
  ~ChunkReader() {
    for (auto& b : buf_) if (b) ngsq_host_free(b);
    if (fd_ >= 0) close(fd_);
  }
  bool direct() const { return direct_; }

  // streams file bytes [lo, hi) (lo on a block boundary) into e.  same_run: e's run already holds the submits of the previous
  // call (an earlier file, before ngsq_next_file), whose copies may still read the buffers.
  void run(ngsq_engine* e, uint64_t lo, uint64_t hi, Progress* progress, bool same_run = false) {
    uint64_t pos = lo & ~uint64_t(4095);  // aligned file position of the next read
    size_t skip = (size_t)(lo - pos);     // bytes of the first read that precede the shard
    size_t carry = 0;                     // bytes of a partial block kept from the previous chunk
    const uint8_t* carry_src = nullptr;
    uint32_t& submits = submits_;         // ngsq_submit calls of e's run so far (ngsq_wait_copied counts them)
    int32_t* used_by = used_by_;          // the submit that last read each buffer
    if (!same_run) {
      submits = 0;
      for (int b = 0; b < kBufs; ++b) used_by[b] = -1;
    }
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
  uint32_t submits_ = 0;
  int32_t used_by_[kBufs] = {-1, -1, -1};
};

// f(i) for every i < n, each in a thread of its own; once all have returned, the first error (the lowest i) is thrown again.
template <class F>
void on_each(size_t n, const F& f) {
  std::vector<std::string> errs(n);
  std::vector<std::thread> ts;
  for (size_t i = 0; i < n; ++i)
    ts.emplace_back([&, i] {
      try {
        f(i);
      } catch (const std::exception& ex) {
        errs[i] = ex.what();
      }
    });
  for (auto& t : ts) t.join();
  for (auto& s : errs) if (!s.empty()) throw std::runtime_error(s);
}

// One engine over its queue of (file, shard) entries: each entry's range and bytes, ngsq_next_file between two entries, one
// ngsq_finish behind the last.  An empty entry sets the range (0, 0) and streams nothing.  A read longer than the
// quality-by-position table (131072 positions by default) sizes the table for the longest read the scan met and runs the
// queue again: the engine keeps nothing of a file it has streamed.  Returns ngsq_finish's code; any other failure throws.
int stream_queue(ngsq_engine* e, const std::vector<FilePart>& queue, const std::vector<std::string>& paths, const std::vector<const MappedFile*>& files,
              size_t chunk_bytes, bool direct, bool log_progress) {
  std::unique_ptr<ChunkReader> reader;  // made at the first live entry: a queue without one allocates no pinned buffers
  for (int attempt = 0;; ++attempt) {
    Progress progress;
    bool same_run = false;  // an earlier entry of this attempt has submitted to e
    for (size_t k = 0; k < queue.size(); ++k) {
      const FilePart& q = queue[k];
      if (k) check(e, ngsq_next_file(e));
      check(e, ngsq_set_range(e, q.shard.first_voffset, q.shard.end_voffset));
      if (q.shard.empty) continue;
      uint64_t lo, hi;
      shard_bytes(q.shard, files[q.file]->data(), files[q.file]->size(), &lo, &hi);
      if (!reader) reader = std::make_unique<ChunkReader>(paths[q.file], chunk_bytes, direct);
      else reader->reopen(paths[q.file], direct);
      reader->run(e, lo, hi, log_progress ? &progress : nullptr, same_run);
      same_run = true;
    }
    const int rc = ngsq_finish(e);
    if (rc == NGSQ_E_QUAL_CAP && attempt == 0) {
      ngsq_stats st;
      check(e, ngsq_get_stats(e, &st));
      info("  [*] Reads of up to " + std::to_string(st.max_read_len) + " bases: enlarging the quality table and reading the " +
           (queue.size() > 1 ? "files" : "file") + " again.");
      check(e, ngsq_reset(e));
      check(e, ngsq_set_quality_positions(e, (uint32_t)st.max_read_len + 1));
      continue;
    }
    if (!rc && log_progress) progress.report(e);
    return rc;
  }
}

// Every engine over its queue, one thread each; only engine 0 logs progress.  When the plan is cut, the shards of a file start
// at record anchors that are speculative until the run proves them.  An anchor is proven when the range in front of it closes
// on it; a file's first record after the header is proven, so the cuts are proven in file order: a part whose start is proven
// and that fails with NGSQ_E_CHAIN or NGSQ_E_TRUNCATED, with a next part of the same file behind it, ends on a false anchor.
// That cut is dropped: the part is run again over both ranges, the next engine over an empty one.  Any other failure is the
// file's and is reported.  On return every engine has finished and the plan holds the ranges that ran.
void run_plan(const std::vector<ngsq_engine*>& engines, FilePlan& plan, const std::vector<std::string>& paths, const std::vector<const MappedFile*>& files,
              size_t chunk_bytes, bool direct) {
  const size_t n = engines.size();
  std::vector<std::string> errs(n);
  std::vector<int> codes(n, 0);
  auto run = [&](size_t i, bool log_progress) {
    try {
      codes[i] = stream_queue(engines[i], plan.queues[i], paths, files, chunk_bytes, direct, log_progress);
      check(engines[i], codes[i]);
    } catch (const std::exception& ex) {
      errs[i] = ex.what();
    }
  };
  on_each(n, [&](size_t i) { run(i, i == 0); });
  for (size_t k = 0; k < n; ++k) {
    while (!errs[k].empty()) {
      if (!plan.cut) throw std::runtime_error(errs[k]);
      const uint32_t f = plan.queues[k][0].file;
      size_t j = k + 1;  // the next live part of the file: its start is the cut in question
      while (j < n && plan.queues[j][0].file == f && plan.queues[j][0].shard.empty) ++j;
      if (j == n || plan.queues[j][0].file != f || (codes[k] != NGSQ_E_CHAIN && codes[k] != NGSQ_E_TRUNCATED)) throw std::runtime_error(errs[k]);
      Shard& part = plan.queues[k][0].shard;
      Shard& next = plan.queues[j][0].shard;
      info("  [*] The record anchor at virtual offset " + std::to_string(next.first_voffset) +
           " is not a record start: dropping that cut and reading the range again.");
      part.end_voffset = next.end_voffset;
      next = Shard();
      next.empty = true;
      for (size_t i : {k, j}) {
        check(engines[i], ngsq_reset(engines[i]));
        errs[i].clear();
        codes[i] = 0;
      }
      check(engines[j], stream_queue(engines[j], plan.queues[j], paths, files, chunk_bytes, direct, false));
      run(k, false);
    }
  }
}

// A one-file ShardPlan as a FilePlan: one entry per device.  cut: the shards start at record anchors found in the file
// (plan_shards_unindexed), which the run proves.
FilePlan file_plan_of(const ShardPlan& p, bool cut) {
  FilePlan plan;
  for (const Shard& s : p.shards) plan.queues.push_back({{0, s}});
  plan.split = p.split;
  plan.cut = cut;
  plan.dropped = p.dropped;
  return plan;
}

// The record anchor finder of plan_shards_unindexed on engine e (after ngsq_set_references)
FindRecord engine_finder(ngsq_engine* e) {
  return [e](const uint8_t* p, size_t n, uint64_t off, uint64_t* voff, int32_t* ref) { check(e, ngsq_find_record(e, p, n, off, voff, ref)); };
}

// The parts' .bai (or uncompressed .csi) of a one-file plan that has run, in file order (engines with an empty range hold no part)
std::vector<uint8_t> join_parts(const std::vector<ngsq_engine*>& engines, const FilePlan& plan, bool csi) {
  std::vector<ngsq_engine*> parts;
  for (size_t i = 0; i < engines.size(); ++i)
    if (!plan.queues[i][0].shard.empty) parts.push_back(engines[i]);
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

void log_dropped_cuts(uint32_t dropped) {
  if (dropped) info("  [*] " + std::to_string(dropped) + " cut(s) left out: no record start found behind the target, or the anchor repeats.");
}

// command.rs:226-421
int app(const QcArgs& args, const ReferenceGenome& genome, const std::string& output_prefix, const std::string& output_directory) {
  // open_and_parse(src, IndexCheck::Full): bam.rs:77-123, for every file of the sample
  std::vector<std::string> paths{args.src};
  paths.insert(paths.end(), args.also.begin(), args.also.end());
  for (const std::string& p : paths)
    if (p.size() < 4 || p.substr(p.size() - 4) != ".bam") throw std::runtime_error("could not open " + p + ": expected a .bam file");
  MappedFile file(args.src);
  std::vector<std::unique_ptr<MappedFile>> also_files;
  for (const std::string& p : args.also) also_files.push_back(std::make_unique<MappedFile>(p));
  const std::string bai_path = args.src + ".bai";  // pathbuf.rs:59-75: x.bam -> x.bam.bai
  const std::string csi_path = args.src + ".csi";  // x.bam -> x.bam.csi: planned from when there is no .bai
  // --cuda-any-order: neither index is read, even when one exists (it may belong to another order of the same records)
  const bool have_bai = !args.any_order && std::filesystem::exists(bai_path), have_csi = !args.any_order && !have_bai && std::filesystem::exists(csi_path);
  // --cuda-build-index: an existing index (.bai, else .csi) is used as it is; a missing one is built by this pass
  const bool build_index = args.build_index && !have_bai && !have_csi;
  const bool build_csi = build_index && args.csi;
  // the .csi is BGZF: it is read once an engine can inflate it (below); without any index read_bai reports the missing .bai
  BaiIndex bai = build_index || have_csi || args.any_order ? BaiIndex{} : read_bai(bai_path);
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
  if (args.by_read_group) flags |= NGSQ_F_READ_GROUPS;  // --only leaves a record facet here (check_read_group_facet)
  if (args.verify_crc) flags |= NGSQ_F_VERIFY_CRC;
  if (build_index) flags |= NGSQ_F_INDEX_PART | (build_csi ? NGSQ_F_INDEX_CSI : 0u);
  if (args.num_records && n_dev > 1) throw std::runtime_error("-n needs a single device (records are counted in file order)");
  // --cuda-by-read-group: the groups are the union of the files' @RG IDs, checked before any device work
  std::vector<std::string> rg_ids;
  if (args.by_read_group) {
    std::vector<std::vector<std::string>> per_file{read_group_ids(bam_header_text(file.data(), file.size(), args.src), args.src)};
    for (size_t k = 0; k < args.also.size(); ++k)
      per_file.push_back(read_group_ids(bam_header_text(also_files[k]->data(), also_files[k]->size(), args.also[k]), args.also[k]));
    rg_ids = union_read_group_ids(per_file);
    info("  [*] " + std::to_string(rg_ids.size()) + " read group" + (rg_ids.size() == 1 ? "" : "s") + ": one more results file each.");
  }
  std::string rg_blob;
  for (const std::string& id : rg_ids) { rg_blob += id; rg_blob += '\0'; }

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
  // --cuda-also: one dictionary for the sample, checked before the qc pass (the genome check below then covers every file)
  std::vector<BamHeader> headers{header};
  std::vector<const MappedFile*> files{&file};
  std::vector<uint64_t> sizes{file.size()};
  std::vector<const uint8_t*> data{file.data()};
  for (size_t k = 0; k < args.also.size(); ++k) {
    headers.push_back(read_bam_header(engines[0], also_files[k]->data(), also_files[k]->size()));
    check_same_dictionary(args.src, header.reference_sequences, args.also[k], headers.back().reference_sequences);
    files.push_back(also_files[k].get());
    sizes.push_back(also_files[k]->size());
    data.push_back(also_files[k]->data());
  }

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

  // every device's queue of (file, shard) entries.  Records in any order (and several files): whole files queued on the devices,
  // or each file cut at record anchors between its devices, every reference split on several devices (plan_files).  Without an
  // index on several devices: the file cut at record anchors (plan_shards_unindexed).  Otherwise contig-aligned file ranges from
  // the index (BAI or CSI), or ranges cut inside contigs when those leave a device idle or unbalanced (choose_shards).  A
  // contig cut between shards is declared on every engine and merged by ngsq_reduce.
  std::vector<uint32_t> ref_len;
  for (auto& rs : header.reference_sequences) ref_len.push_back(rs.length);
  const bool several_files = !args.also.empty();
  FindRecord find;  // the anchor finder needs the references (every engine sets them again below)
  if (n_dev > 1 && (args.any_order || build_index)) {
    check(engines[0], ngsq_set_references(engines[0], (uint32_t)ref_len.size(), ref_len.data(), std::vector<uint8_t>(ref_len.size(), 0).data()));
    find = engine_finder(engines[0]);
  }
  FilePlan plan;
  if (args.any_order) {
    plan = plan_files(headers, data, sizes, n_dev, find);
    log_dropped_cuts(plan.dropped);
    if (several_files)
      info("  [*] " + std::to_string(paths.size()) + " files of one sample" +
           (n_dev == 1 ? std::string(" on one device.")
                       : std::string(plan.cut ? ", each cut between its devices" : ", whole files queued on the devices") + ", every reference split."));
    else if (n_dev > 1)
      info("  [*] Records in any order: " + std::to_string(n_dev - plan.dropped) + " shards, every reference split.");
  } else {
    const bool cut = build_index && n_dev > 1;
    const ShardPlan p = cut ? plan_shards_unindexed(header, file.data(), file.size(), n_dev, find) : choose_shards(header, bai, n_dev, file.size());
    log_dropped_cuts(p.dropped);
    if (p.split_plan) {
      std::string names;
      for (uint32_t c : p.split) names += (names.empty() ? "" : ", ") + header.reference_sequences[c].name;
      info("  [*] Sharding inside contigs: " + std::to_string(n_dev) + " shards" + (names.empty() ? std::string() : ", split: " + names) + ".");
    }
    plan = file_plan_of(p, cut);
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
    if (args.by_read_group) check(engines[i], ngsq_set_read_groups(engines[i], (uint32_t)rg_ids.size(), rg_blob.data(), rg_blob.size()));
  }
  if (n_dev > 1) {
    char id[128];
    if (ngsq_nccl_unique_id(id)) throw std::runtime_error(std::string("NCCL: ") + ngsq_last_error(nullptr));
    on_each(n_dev, [&](size_t i) {
      if (ngsq_comm_init(engines[i], (int)n_dev, (int)i, id)) throw std::runtime_error(std::string("NCCL: ") + ngsq_last_error(engines[i]));
    });
  }

  // the hot path: one thread per GPU
  info("Starting CUDA pass for QC stats.");
  const auto t_hot = std::chrono::steady_clock::now();
  run_plan(engines, plan, paths, files, args.chunk_mb << 20, args.direct_io);
  if (n_dev > 1)
    on_each(n_dev, [&](size_t i) { if (ngsq_reduce(engines[i], 0)) throw std::runtime_error(std::string("NCCL: ") + ngsq_last_error(engines[i])); });
  // the index of this pass: joined (and its order checked) before any output is written
  std::vector<uint8_t> new_index;
  if (build_index) new_index = join_parts(engines, plan, build_csi);
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
  if (args.by_read_group) {
    const uint64_t ungrouped = write_read_group_results(root, rg_ids, genome, args.only_facet, output_prefix, output_directory);
    if (ungrouped)
      std::cerr << "WARN " << ungrouped << " record(s) carry no RG tag, or one that no @RG line declares: written to "
                << no_read_group_prefix(output_prefix) << ".results.json\n";
  }
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
         << ",\"ms_total\":" << st.ms_total << ",\"ms_tail\":" << st.ms_tail << ",\"waves\":" << st.waves << ",\"wall_ms_file_to_results\":" << hot_ms;
      if (several_files) {
        uint32_t n_files = 0;
        for (const FilePart& q : plan.queues[i]) n_files += q.shard.empty ? 0 : 1;
        pf << ",\"files\":" << n_files;
      }
      pf << "}";
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

// `ngs index` for a BAM (src/index/bam.rs:39-109): the header, then every record through the engines' NGSQ_F_INDEX_PART pass,
// and the .bai next to the file (utils/pathbuf.rs:59-75: x.bam -> x.bam.bai).  Like the reference (bam.rs:52-58) it never
// overwrites an existing index.  On several devices the file is cut at record anchors, one engine and one thread per part,
// and the parts are joined on the host; one device indexes one part from the first record to EOF.  No collective is involved,
// so a device may repeat.
struct IndexArgs {
  std::string src;
  bool csi = false;          // --csi: <BAM>.csi (BGZF) instead of <BAM>.bai
  uint32_t min_shift = 14;   // -m / --min-shift (CSI); the depth follows samtools' rule
  int device = 0;            // --cuda-device: the one device when --cuda-devices names none
  std::vector<int> devices;  // --cuda-devices: several engines, one part of the file each
  bool verify_crc = true;
  size_t chunk_mb = 64;
  bool direct_io = true;
};

int index_command(const IndexArgs& a) {
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
  const ShardPlan p = plan_shards_unindexed(header, file.data(), file.size(), (uint32_t)n_dev, engine_finder(engines[0]));
  log_dropped_cuts(p.dropped);
  info(n_dev == 1 ? std::string("Indexing BAM file.") : "Indexing BAM file in " + std::to_string(n_dev - p.dropped) + " parts.");
  FilePlan plan = file_plan_of(p, true);
  run_plan(engines, plan, {a.src}, {&file}, a.chunk_mb << 20, a.direct_io);
  uint64_t records = 0;
  for (auto* e : engines) { ngsq_stats st; check(e, ngsq_get_stats(e, &st)); records += st.records; }
  info("Processed " + std::to_string(records) + " records.");
  const std::vector<uint8_t> payload = join_parts(engines, plan, a.csi);
  write_index(dst, a.csi ? bgzf_compress(payload) : payload);  // the .csi is BGZF
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
  if (a.devices.empty()) a.devices = {a.device};
  return index_command(a);
}

void usage() {
  std::cerr << "usage: ngs-cuda-qc qc <BAM> <REFERENCE_GENOME> [-n N] [-o DIR] [-p PREFIX] [--only FACET]\n"
               "                  [--cuda-devices 0,1,..] [--cuda-build-index [--cuda-csi [--cuda-min-shift N]] | --cuda-any-order]\n"
               "                  [--cuda-gc-seed S] [--cuda-no-crc] [--cuda-chunk-mb M] [--cuda-buffered-io] [--cuda-perf]\n"
               "                  (the index is <BAM>.bai, or <BAM>.csi when there is no .bai; --cuda-build-index: without either,\n"
               "                  build <BAM>.bai, or with --cuda-csi <BAM>.csi (min_shift N, default 14), in the same pass and write it\n"
               "                  once the run succeeded; --cuda-any-order: read no index and take the records in any order, not\n"
               "                  with -n, --cuda-build-index or --cuda-csi)\n"
               "       ngs-cuda-qc qc <BAM> <REFERENCE_GENOME> --cuda-also <BAM> [--cuda-also <BAM> ..] [the options above]\n"
               "                  (the records of every file are checked as one sample: the files must have the same reference\n"
               "                  sequences; the rules of --cuda-any-order apply; the output prefix is the first <BAM>'s name)\n"
               "       ngs-cuda-qc qc <BAM> <REFERENCE_GENOME> --cuda-by-read-group [the options above]\n"
               "                  (also writes <PREFIX>.read_group.<ID>.results.json for every @RG line, with General, Template Length,\n"
               "                  GC Content and Quality Score of that group's records, and <PREFIX>.no_read_group.results.json for\n"
               "                  records of no declared group; <ID> with bytes outside [A-Za-z0-9._-] and '%' as %XX; not with\n"
               "                  --only Coverage, Edits or \"Genomic Features\")\n"
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
      else if (s == "--cuda-any-order") a.any_order = true;
      else if (s == "--cuda-also") a.also.push_back(val());
      else if (s == "--cuda-by-read-group") a.by_read_group = true;
      else if (s == "--cuda-min-shift") { a.min_shift = (uint32_t)std::stoul(val()); min_shift_set = true; }
      else if (s == "--cuda-buffered-io") a.direct_io = false;
      else if (s == "-h" || s == "--help") { usage(); return 0; }
      else if (!s.empty() && s[0] == '-' && s != "-") throw std::runtime_error("unknown flag " + s);
      else pos.push_back(s);
    }
    if (pos.size() != 2 || a.devices.empty()) { usage(); return 2; }
    if (!a.also.empty()) {
      if (a.num_records)
        throw std::runtime_error("--cuda-also cannot be combined with -n: the first N records are counted in the order of one file");
      if (a.build_index) throw std::runtime_error("--cuda-also cannot be combined with --cuda-build-index: an index describes one file");
      if (a.csi) throw std::runtime_error("--cuda-also cannot be combined with --cuda-csi: an index describes one file");
      a.any_order = true;  // a file boundary is one more cut: records of several files come in no common order
    }
    if (a.any_order && a.num_records)
      throw std::runtime_error("--cuda-any-order cannot be combined with -n: the first N records are counted in the order of the per-contig "
                               "queries, which records in any order do not have");
    if (a.any_order && a.build_index) throw std::runtime_error("--cuda-any-order cannot be combined with --cuda-build-index: an index needs coordinate-sorted records");
    if (a.any_order && a.csi) throw std::runtime_error("--cuda-any-order cannot be combined with --cuda-csi: an index needs coordinate-sorted records");
    if (a.build_index && a.num_records) throw std::runtime_error("--cuda-build-index cannot be combined with -n: an index covers every record of the file");
    if (a.csi && !a.build_index) throw std::runtime_error("--cuda-csi sets the format of the index --cuda-build-index writes: use it with --cuda-build-index");
    if (min_shift_set && !a.csi) throw std::runtime_error("--cuda-min-shift sets the binning of a CSI: use it with --cuda-csi");
    if (a.by_read_group) check_read_group_facet(a.only_facet);
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
