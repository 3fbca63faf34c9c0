// libngs_cuda.so — implementation of include/ngs_cuda.h.
// One engine = one GPU = one host thread.  The file is STREAMED: blocks are inflated in waves (one launch of the
// decode kernel each) into two recycled slots, and every wave's records are scanned and tallied before its slot is
// reused, so the device footprint does not grow with the file (30x WGS, 270 GB inflated, runs in a few GB):
//   compressed staging ring | 2 x [headroom | one wave of inflated bytes] | match bitmap of a wave | per-wave block
//   tables | record offset table of a wave (8 B/record) | per-contig int32 difference arrays | packed u64 result
//   buffer (the NCCL payload) | RunState (everything that links two waves, recscan.cuh).
// Streams: H2D copies on s_copy; inflate (decode + resolve) on s_comp; record scan + facet kernels on s_scan, beside the
// inflate of the NEXT wave (the decoder owns the SMs' shared memory but leaves room for the scan kernels; the facet kernels
// share the SMs with the resolve kernel); the per-block CRC32 check on s_aux, enqueued behind the start of the next
// wave's decode.  A wave is enqueued without any host round trip: the submitting thread never waits for the GPU, the PCIe
// copy of chunk k+1 overlaps the kernels of wave k, and after the last chunk has arrived only the last (small) wave,
// the coverage resolve and the result read-back remain.
#include <dlfcn.h>
#include <time.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include <cuda_runtime.h>

#include "../../include/ngs_cuda.h"
#include "cov_n.cuh"
#include "coverage.cuh"
#include "crc32.cuh"
#include "edits.cuh"
#include "facets.cuh"
#include "features.cuh"
#include "index.cuh"
#include "inflate2.cuh"
#include "read_groups.cuh"
#include "recscan.cuh"

using namespace ngsq;

namespace {

thread_local std::string g_create_err;

struct NcclApi {
  void* lib = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  void* CommInitRank = nullptr;  // ncclCommInitRank(ncclComm_t*, int, ncclUniqueId by value, int)
  int (*Reduce)(const void*, void*, size_t, int, int, int, void*, cudaStream_t) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
struct NcclId { char b[128]; };

NcclApi g_nccl;
bool load_nccl(std::string& err) {
  if (g_nccl.lib) return true;
  const char* names[] = {"libnccl.so.2", "libnccl.so"};
  for (const char* n : names) {
    g_nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
    if (g_nccl.lib) break;
  }
  if (!g_nccl.lib) { err = std::string("cannot load libnccl: ") + dlerror(); return false; }
  auto sym = [&](const char* s) { return dlsym(g_nccl.lib, s); };
  g_nccl.GetUniqueId = (int (*)(void*))sym("ncclGetUniqueId");
  g_nccl.CommInitRank = sym("ncclCommInitRank");
  g_nccl.Reduce = (int (*)(const void*, void*, size_t, int, int, int, void*, cudaStream_t))sym("ncclReduce");
  g_nccl.AllReduce = (int (*)(const void*, void*, size_t, int, int, void*, cudaStream_t))sym("ncclAllReduce");
  g_nccl.CommDestroy = (int (*)(void*))sym("ncclCommDestroy");
  g_nccl.GetErrorString = (const char* (*)(int))sym("ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.Reduce || !g_nccl.AllReduce) {
    err = "libnccl is missing symbols";
    return false;
  }
  return true;
}

}  // namespace

// NGSQ_F_INDEX / NGSQ_F_INDEX_PART: an engine's index state on the host once its last wave is done.  Every part is linear or
// order-free, so the state of parts cut from one file joins exactly (ngsq_join_bai / ngsq_join_csi): runs and overflow lists
// concatenate, windows take the minimum, maxw the maximum, counts and n_no_coor add up.
struct IxHost {
  IndexState S{};
  std::vector<IndexRun> runs;       // in any order (ix_collect sorts them)
  std::vector<IndexOvf> ovf;        // the overflow list, BAI entries unpacked
  std::vector<uint64_t> win, counts;
  std::vector<uint32_t> maxw;
  uint64_t last_order_key = 0;      // of the part's last record that constrains the order (0 = none)
  uint64_t data_end = 0;            // virtual offset behind the last record submitted
};

struct ngsq_engine {
  int device = 0;
  int n_sm = 0;
  ngsq_config cfg{};
  std::string err;
  cudaStream_t s_copy = nullptr, s_comp = nullptr, s_scan = nullptr, s_aux = nullptr;
  cudaEvent_t ev_start = nullptr, ev_a = nullptr, ev_b = nullptr, ev_d = nullptr, ev_e = nullptr, ev_f = nullptr, ev_g = nullptr;
  bool run_started = false, finished = false;

  // references / coverage
  uint32_t n_ref = 0;
  std::vector<uint32_t> ref_len;
  std::vector<uint8_t> cov_enabled;
  std::vector<uint64_t> diff_base;
  std::vector<uint32_t> cov_slot, cov_nbins;
  uint32_t* d_ref_len = nullptr;
  uint8_t* d_cov_enabled = nullptr;
  uint64_t* d_diff_base = nullptr;
  uint32_t* d_cov_slot = nullptr;
  int32_t* d_diff = nullptr;
  uint64_t diff_elems = 0;
  int64_t* d_tile = nullptr;         // tile bases of the contig being resolved
  uint32_t tile_cap = 0;
  std::vector<uint32_t> tile_off;    // first tile of every contig in d_tile_sum
  uint32_t* d_tile_off = nullptr;
  int32_t* d_tile_sum = nullptr;     // sums of the difference arrays per 4096-position tile, maintained by the scatter
  uint64_t tile_total = 0;
  bool trace = false;                // NGSQ_TRACE=1: per-wave and per-chunk timeline on stderr at ngsq_finish
  std::vector<double> host_ms;       // host clock at every wave launch (trace)
  double host_t0 = 0;

  // results: [fixed | per-contig coverage slots | quality table, qpos_cap rows]
  uint64_t* d_res = nullptr;
  LongRead* d_long = nullptr;        // the wave's reads longer than the facet kernel's shared-memory quality tables
  uint64_t long_cap = 0;
  size_t res_words = 0, res_cap_words = 0;
  uint32_t qual_off = R_FIXED_WORDS;
  uint32_t qpos_cap = 0;
  uint32_t qpos_dirty = 0;  // quality rows an earlier run may have written (zeroed at the next start)
  std::vector<uint64_t> h_res;
  uint32_t h_qpos = 0;

  // submitted blocks (host tables for the whole run; the device only ever sees one wave)
  std::vector<BlockDesc> h_blocks;  // in_off absolute, out_off = inflated offset in the whole stream
  std::vector<uint32_t> h_crc;
  uint64_t out_used = 0;            // inflated bytes submitted so far
  uint64_t comp_bytes_total = 0;
  struct Chunk { cudaEvent_t copied; uint32_t blocks_end; };
  std::vector<Chunk> chunks;        // host submits: blocks [.., blocks_end) are on the device once `copied` fired
  uint32_t launched = 0;            // blocks [0, launched) have been handed to a wave

  // compressed staging ring
  struct CompSeg { uint8_t* ptr; size_t cap, used; uint32_t blocks_end; };
  std::vector<CompSeg> comp_segs;
  size_t comp_total = 0;

  // waves
  struct Wave { cudaEvent_t begin, decoded_from, decoded, resolved, scan_begin, begun, scan_end, facets_end, crc_begin, crc_end; uint32_t b0, b1; bool scanned, crc_launched; const uint8_t* out; };
  std::vector<Wave> waves;
  uint32_t headroom = 0;
  uint8_t* d_slot[2] = {nullptr, nullptr};
  size_t slot_cap[2] = {0, 0};       // data bytes behind the headroom
  // block descriptors and expected CRCs of the whole run, uploaded behind each chunk ON THE COPY STREAM: a wave's
  // tables are on the device when its bytes are, and no other stream ever queues a copy behind the chunk copies
  BlockDesc* d_blocks_all = nullptr;
  uint32_t* d_crc_all = nullptr;
  uint32_t blocks_all_cap = 0;
  struct PinSlab { uint8_t* p; size_t cap, used; };
  std::vector<PinSlab> pin_slabs;    // pinned staging of those uploads (lives until ngsq_reset)
  uint32_t *d_wstatus[2] = {nullptr, nullptr}, *d_first = nullptr, *d_landed = nullptr, *d_count = nullptr;
  uint64_t* d_base = nullptr;
  uint32_t scan_cap = 0;
  uint32_t* d_bitmap = nullptr;
  size_t bitmap_cap = 0;             // blocks
  uint64_t* d_rec = nullptr;
  uint64_t rec_cap = 0;
  uint32_t* d_mark = nullptr;
  uint64_t mark_cap = 0;
  uint32_t* d_queue = nullptr;
  RunState* d_state = nullptr;
  RunState* h_state = nullptr;       // pinned
  uint64_t* h_prog = nullptr;        // pinned ring: {rec_base, wave_rec} after each wave's scan (ngsq_progress)
  uint32_t prog_seen = 0;            // waves whose probe has been consumed
  uint64_t prog_records = 0;
  CrcTables* d_crc_tables = nullptr;

  // shard range (virtual offsets -> blocks, resolved as the blocks arrive)
  uint64_t first_voff = 0, end_voff = 0;
  bool range_set = false, start_resolved = false, end_resolved = false;
  uint32_t start_block = 0, start_uo = 0, end_block = 0, end_uo = 0;
  // several files in one run (ngsq_next_file): the current file's blocks are [file_b0, ..); between ngsq_next_file and the
  // next ngsq_set_range no chunk may be submitted
  uint32_t file_b0 = 0;
  bool awaiting_range = false;

  ngsq_stats stats{};
  uint32_t other_launches = 0;
  size_t facet_smem = 0;
  int facet_occ = 0;

  // Edits facet (NGSQ_F_EDITS): per-contig FASTA codes, per-position counters, result block
  std::vector<EditsContig> ed_contigs;
  std::vector<void*> ed_allocs;          // device allocations behind ed_contigs
  EditsContig* d_ed_contigs = nullptr;
  uint32_t *d_ed_refs = nullptr, *d_ed_alts = nullptr;
  uint64_t ed_pos_total = 0;
  unsigned long long* d_ed_res = nullptr;
  std::vector<uint64_t> h_ed_res;

  // Genomic Features facet (NGSQ_F_FEATURES): per contig and class, sorted starts / stops; nine counters
  std::vector<FeatureContig> ft_contigs;
  std::vector<void*> ft_allocs;
  FeatureContig* d_ft_contigs = nullptr;
  uint8_t ft_slot_class[8] = {0, 1, 2, 3, 4, 0, 0, 0};
  bool ft_model_set = false;
  unsigned long long* d_ft_res = nullptr;
  std::vector<uint64_t> h_ft_res;

  // BAI build (NGSQ_F_INDEX): per-reference linear-index tables and counters for the whole run; per indexed wave a run table
  // (two, by parity), drained to pinned host memory when the wave two later is launched
  IndexState* d_ix = nullptr;
  IndexRun* d_ix_runs[2] = {nullptr, nullptr};
  uint64_t ix_runs_cap = 0;
  void* d_ix_ovf = nullptr;          // IndexRun entries (BAI) or IndexOvf entries (CSI)
  uint64_t* d_ix_win_base = nullptr;
  uint32_t* d_ix_win_n = nullptr;
  unsigned long long* d_ix_win = nullptr;
  unsigned int* d_ix_maxw = nullptr;
  unsigned long long* d_ix_counts = nullptr;
  std::vector<uint64_t> ix_win_base;
  std::vector<uint32_t> ix_win_n;
  uint64_t ix_win_total = 0;
  uint64_t* h_ix_probe = nullptr;    // pinned: run count of the wave in slot 0 / 1
  struct IxWave { cudaEvent_t done; bool drained; };
  std::vector<IxWave> ix_waves;
  std::vector<std::pair<const IndexRun*, uint64_t>> ix_drained;  // pinned copies of drained run tables
  uint64_t data_end_coff = 0;        // end of the last non-empty block submitted (the offset after the last record)
  std::vector<uint8_t> ix_bytes;     // the .bai, or the uncompressed .csi (NGSQ_F_INDEX_CSI)
  IxHost ix;                         // NGSQ_F_INDEX_PART: the part's state for ngsq_join_bai / ngsq_join_csi
  // NGSQ_F_INDEX_CSI: the binning asked for (ngsq_set_index_binning; depth 0 = samtools' rule) and the one in use, resolved
  // by ngsq_set_references from the longest reference; kept across ngsq_reset
  uint32_t ix_min_shift = kIxWindowShift, ix_depth_req = 0, ix_depth = 5;
  bool ix_part_ok = false;           // ... valid: ngsq_finish succeeded

  // references split between shards (ngsq_split_reference): scattered as usual, resolved only by the merge
  std::vector<uint8_t> split_ref;
  uint32_t n_split = 0;
  bool split_merged = false;         // the split references of this run have been merged (reduce / resolve_split)

  // read groups (NGSQ_F_READ_GROUPS): the IDs, their device hash table, the group buffer
  // [sums (rg_n + 1) x kGroupSums | quality lengths (rg_n + 1) | quality tables (rg_n + 1) x grp_rows x 94], the per-wave
  // bucketing arrays, and the host copies ngsq_select_read_group serves
  bool rg_set = false;
  uint32_t rg_n = 0, rg_mask = 0;
  uint64_t rg_sig = 0;               // hash of the IDs and their number (part of ngsq_reduce's layout agreement)
  uint8_t* d_rg_ids = nullptr;
  uint32_t *d_rg_id_off = nullptr, *d_rg_table = nullptr;
  uint64_t* d_grp = nullptr;
  uint32_t grp_rows = 0, grp_dirty = 0;  // rows of each group table; rows an earlier run may have written
  uint16_t* d_rg_of = nullptr;
  uint32_t *d_rg_order = nullptr, *d_rg_count = nullptr, *d_rg_cursor = nullptr, *d_rg_total = nullptr;
  uint64_t rg_cap = 0;               // records the bucketing arrays hold
  size_t rg_smem = 0;
  int rg_occ = 1;
  std::vector<uint64_t> h_grp_sums, h_grp_qlen;
  std::vector<std::vector<uint64_t>> h_grp_qual;
  int32_t rg_sel = -1;

  // nccl
  void* comm = nullptr;
  int n_ranks = 1, rank = 0;
  bool layout_agreed = false;
};

namespace {

constexpr uint32_t kDefaultHeadroom = 16u << 20;       // longest record that may straddle two waves
constexpr uint32_t kDefaultQualPositions = 1u << 17;   // rows of the global quality table (98 MB)
constexpr uint32_t kProgSlots = 1024;
constexpr size_t kDefaultCompRing = (size_t)8 << 30;   // compressed staging kept on the device when the caller reserves nothing
constexpr uint64_t kIndexOverflowCap = 1u << 20;       // records that reach past their reference's linear-index table

int fail(ngsq_engine* e, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (e) e->err = buf; else g_create_err = buf;
  return code;
}

#define CU(call)                                                                                       \
  do {                                                                                                 \
    cudaError_t _rc = (call);                                                                          \
    if (_rc != cudaSuccess) return fail(e, NGSQ_E_CUDA, "%s: %s (%s:%d)", #call, cudaGetErrorString(_rc), __FILE__, __LINE__); \
  } while (0)

// (re)allocates a device buffer that holds no live data; the caller has made sure nothing in flight uses it
template <class T>
int fresh(ngsq_engine* e, T*& ptr, size_t n, const char* what) {
  if (ptr) cudaFree(ptr);
  ptr = nullptr;
  cudaError_t rc = cudaMalloc(&ptr, n * sizeof(T));
  if (rc != cudaSuccess) return fail(e, NGSQ_E_NOMEM, "cudaMalloc %s (%zu bytes): %s", what, n * sizeof(T), cudaGetErrorString(rc));
  return NGSQ_OK;
}

uint32_t wave_blocks(const ngsq_engine* e) { return (uint32_t)e->n_sm * kDecThreads; }

// the K13 index pass runs: a whole file (NGSQ_F_INDEX) or one part of it (NGSQ_F_INDEX_PART)
bool ix_on(const ngsq_engine* e) { return e->cfg.flags & (NGSQ_F_INDEX | NGSQ_F_INDEX_PART); }
// ... and builds a CSI instead of a BAI
bool ix_csi(const ngsq_engine* e) { return e->cfg.flags & NGSQ_F_INDEX_CSI; }

uint32_t launch_quantum(const ngsq_engine* e) {
  // One wave = one block per decoder lane: a launch takes about one block-decode latency whatever its size (every
  // lane decodes its block serially), so smaller launches only add latencies.  When the caller announced the number
  // of blocks (reserve_blocks), the waves are made equal.
  if (e->cfg.launch_blocks) return e->cfg.launch_blocks;
  const uint32_t wave = wave_blocks(e);
  if (e->cfg.reserve_blocks > wave) {
    const uint32_t n_waves = (e->cfg.reserve_blocks + wave - 1) / wave;
    return (e->cfg.reserve_blocks + n_waves - 1) / n_waves;
  }
  return wave;
}

int layout_results(ngsq_engine* e, uint32_t qpos) {
  // fixed | per-contig coverage slots | quality table (last, so that its size may differ per engine)
  uint32_t off = R_FIXED_WORDS;
  e->cov_slot.assign(e->n_ref, 0);
  e->cov_nbins.assign(e->n_ref, 0);
  for (uint32_t c = 0; c < e->n_ref; ++c) {
    e->cov_slot[c] = off;
    if (e->cov_enabled[c]) {
      uint32_t L = e->ref_len[c];
      uint32_t nb = 1 + L / kCovBin + (L % kCovBin ? 1 : 0);
      e->cov_nbins[c] = nb;
      off += COV_BINS + nb + 1;
    }
  }
  e->qual_off = off;
  e->qpos_cap = qpos;
  e->res_words = (size_t)off + (size_t)qpos * 94;
  return NGSQ_OK;
}

bool rg_on(const ngsq_engine* e) { return e->cfg.flags & NGSQ_F_READ_GROUPS; }

// The group buffer for `rows` quality rows per group (layout: see ngsq_engine::d_grp).  keep: the counters and the quality
// rows a finished run wrote move into the new buffer.  Only between runs.
int alloc_groups(ngsq_engine* e, uint32_t rows, bool keep) {
  const uint64_t ng = (uint64_t)e->rg_n + 1, head = ng * (kGroupSums + 1), words = head + ng * rows * 94;
  uint64_t* np = nullptr;
  cudaError_t rc = cudaMalloc(&np, words * 8);
  if (rc != cudaSuccess) {
    cudaGetLastError();
    return fail(e, NGSQ_E_NOMEM, "read-group tables: %llu groups (%u read groups + ungrouped) with %u quality rows each need %.1f GB of device memory "
                "(ngsq_set_read_groups sets the groups, ngsq_set_quality_positions the rows): %s",
                (unsigned long long)ng, e->rg_n, rows, words * 8 / 1e9, cudaGetErrorString(rc));
  }
  CU(cudaMemsetAsync(np, 0, words * 8, e->s_comp));
  if (keep && e->d_grp) {
    const uint32_t old = e->grp_rows, copy = std::min(old, rows);
    CU(cudaMemcpyAsync(np, e->d_grp, head * 8, cudaMemcpyDeviceToDevice, e->s_comp));
    if (copy) CU(cudaMemcpy2DAsync(np + head, (size_t)rows * 94 * 8, e->d_grp + head, (size_t)old * 94 * 8, (size_t)copy * 94 * 8, ng,
                                   cudaMemcpyDeviceToDevice, e->s_comp));
  }
  CU(cudaStreamSynchronize(e->s_comp));
  if (e->d_grp) cudaFree(e->d_grp);
  e->d_grp = np;
  e->grp_rows = rows;
  e->grp_dirty = keep ? e->grp_dirty : 0;
  return NGSQ_OK;
}

// Result buffer with room for `qpos` quality rows.  Only between runs (or after ngsq_finish): nothing is in flight.
int ensure_res(ngsq_engine* e, uint32_t qpos, bool keep) {
  if (qpos < 256) qpos = 256;
  if (qpos <= e->qpos_cap && e->d_res) return NGSQ_OK;
  size_t old_words = e->res_words;
  layout_results(e, qpos);
  if (e->res_words > e->res_cap_words) {
    uint64_t* np = nullptr;
    size_t ncap = e->res_words;
    cudaError_t rc = cudaMalloc(&np, ncap * 8);
    if (rc != cudaSuccess) return fail(e, NGSQ_E_NOMEM, "cudaMalloc results (%zu bytes): %s", ncap * 8, cudaGetErrorString(rc));
    CU(cudaMemsetAsync(np, 0, ncap * 8, e->s_comp));
    if (keep && e->d_res && old_words) CU(cudaMemcpyAsync(np, e->d_res, old_words * 8, cudaMemcpyDeviceToDevice, e->s_comp));
    CU(cudaStreamSynchronize(e->s_comp));
    if (e->d_res) cudaFree(e->d_res);
    e->d_res = np;
    e->res_cap_words = ncap;
    e->layout_agreed = false;  // the layout word carries the table's capacity
  }
  if (e->d_cov_slot) CU(cudaMemcpyAsync(e->d_cov_slot, e->cov_slot.data(), e->n_ref * 4, cudaMemcpyHostToDevice, e->s_comp));
  CU(cudaStreamSynchronize(e->s_comp));
  if (e->rg_set && e->grp_rows != e->qpos_cap) return alloc_groups(e, e->qpos_cap, keep);  // a group table has the sample's rows
  return NGSQ_OK;
}

int start_run(ngsq_engine* e) {
  if (e->run_started) return NGSQ_OK;
  if (!e->d_res) { int rc = ensure_res(e, e->cfg.quality_positions ? e->cfg.quality_positions : kDefaultQualPositions, false); if (rc) return rc; }
  CU(cudaEventRecord(e->ev_start, e->s_comp));
  // the fixed part, the coverage slots and every quality row an earlier run may have touched
  const size_t dirty = std::min<size_t>(e->res_words, (size_t)e->qual_off + (size_t)std::max<uint32_t>(e->qpos_dirty, 256) * 94);
  CU(cudaMemsetAsync(e->d_res, 0, dirty * 8, e->s_comp));
  if ((e->cfg.flags & NGSQ_F_COVERAGE) && e->diff_elems) {
    CU(cudaMemsetAsync(e->d_diff, 0, e->diff_elems * 4, e->s_comp));
    CU(cudaMemsetAsync(e->d_tile_sum, 0, e->tile_total * 4, e->s_comp));
  }
  memset(e->h_state, 0, sizeof(RunState));
  e->h_state->bad_block = ~0ull;
  e->h_state->next_carry = kNoCarry;
  CU(cudaMemcpyAsync(e->d_state, e->h_state, sizeof(RunState), cudaMemcpyHostToDevice, e->s_comp));
  if ((e->cfg.flags & NGSQ_F_FEATURES) && e->d_ft_res) CU(cudaMemsetAsync(e->d_ft_res, 0, F_WORDS * 8, e->s_comp));
  if (rg_on(e)) {
    if (!e->rg_set) return fail(e, NGSQ_E_ARG, "NGSQ_F_READ_GROUPS needs ngsq_set_read_groups before the first submit");
    // the counters, the lengths, and every quality row an earlier run may have touched
    const uint64_t ng = (uint64_t)e->rg_n + 1, head = ng * (kGroupSums + 1);
    CU(cudaMemsetAsync(e->d_grp, 0, head * 8, e->s_comp));
    const uint32_t dirty = std::min(e->grp_dirty, e->grp_rows);
    if (dirty) CU(cudaMemset2DAsync(e->d_grp + head, (size_t)e->grp_rows * 94 * 8, 0, (size_t)dirty * 94 * 8, ng, e->s_comp));
    e->grp_dirty = e->grp_rows;  // until ngsq_finish knows better
    CU(cudaMemsetAsync(e->d_rg_count, 0, ng * 4, e->s_comp));
  }
  if (ix_on(e)) {
    if (!e->d_ix) return fail(e, NGSQ_E_ARG, "NGSQ_F_INDEX needs ngsq_set_references before the first submit");
    IndexState z{};
    z.carry[0].run_key = kIxNoRun;
    z.unsorted_voff = ~0ull;
    z.first_key = z.first_voff = ~0ull;
    CU(cudaMemcpyAsync(e->d_ix, &z, sizeof z, cudaMemcpyHostToDevice, e->s_comp));
    if (e->ix_win_total) CU(cudaMemsetAsync(e->d_ix_win, 0xFF, e->ix_win_total * 8, e->s_comp));
    if (e->n_ref) {
      CU(cudaMemsetAsync(e->d_ix_maxw, 0, (size_t)e->n_ref * 4, e->s_comp));
      CU(cudaMemsetAsync(e->d_ix_counts, 0, (size_t)e->n_ref * 16, e->s_comp));
    }
  }
  if ((e->cfg.flags & NGSQ_F_EDITS) && e->d_ed_res) {
    CU(cudaMemsetAsync(e->d_ed_res, 0, E_WORDS * 8, e->s_comp));
    if (e->ed_pos_total) {
      CU(cudaMemsetAsync(e->d_ed_refs, 0, e->ed_pos_total * 4, e->s_comp));
      CU(cudaMemsetAsync(e->d_ed_alts, 0, e->ed_pos_total * 4, e->s_comp));
    }
  }
  // the pinned state block is reused for the read-back at the end: the upload above must have left it
  CU(cudaStreamSynchronize(e->s_comp));
  e->run_started = true;
  return NGSQ_OK;
}

int append_blocks(ngsq_engine* e, const ngsq_block* blk, uint32_t n, uint64_t dev_base_addr, uint64_t first_coffset) {
  for (uint32_t i = 0; i < n; ++i) {
    const ngsq_block& b = blk[i];
    if (b.csize < b.hdr_len + 8 || b.isize > 65536) return fail(e, NGSQ_E_BAD_BLOCK, "malformed BGZF block at file offset %llu", (unsigned long long)b.coffset);
    if (b.isize == 0) continue;  // empty blocks (incl. the EOF marker) carry nothing
    if (e->h_blocks.size() > e->file_b0 && b.coffset <= e->h_blocks.back().coff) return fail(e, NGSQ_E_ARG, "chunks must be submitted in file order (block at file offset %llu)", (unsigned long long)b.coffset);
    BlockDesc d;
    d.in_off = dev_base_addr + (b.coffset - first_coffset) + b.hdr_len;
    d.out_off = e->out_used;
    d.clen = b.csize - b.hdr_len - 8;
    d.isize = b.isize;
    d.coff = b.coffset;
    e->h_blocks.push_back(d);
    e->h_crc.push_back(b.crc32);
    e->out_used += b.isize;
    e->data_end_coff = b.coffset + b.csize;
  }
  return NGSQ_OK;
}

// pinned bytes that stay put until ngsq_reset
void* pin_alloc(ngsq_engine* e, size_t bytes) {
  bytes = (bytes + 63) & ~size_t(63);
  for (auto& ps : e->pin_slabs)
    if (ps.used + bytes <= ps.cap) { void* r = ps.p + ps.used; ps.used += bytes; return r; }
  const size_t cap = std::max<size_t>(bytes, (size_t)8 << 20);
  uint8_t* p = nullptr;
  if (cudaHostAlloc((void**)&p, cap, cudaHostAllocDefault) != cudaSuccess) return nullptr;
  e->pin_slabs.push_back({p, cap, bytes});
  return p;
}

// Descriptors and expected CRCs of blocks [first, end) follow their chunk on the copy stream.
int upload_descriptors(ngsq_engine* e, uint32_t first, uint32_t end) {
  if (end <= first) return NGSQ_OK;
  if (end > e->blocks_all_cap) {
    // the table is sized by reserve_blocks; without it, it doubles (rare: everything in flight is awaited first)
    CU(cudaStreamSynchronize(e->s_copy));
    CU(cudaStreamSynchronize(e->s_comp));
    CU(cudaStreamSynchronize(e->s_scan));
    CU(cudaStreamSynchronize(e->s_aux));
    const uint32_t cap = std::max<uint32_t>(end + end / 2, std::max<uint32_t>(e->cfg.reserve_blocks, 1u << 18));
    BlockDesc* nb = nullptr;
    uint32_t* nc = nullptr;
    if (cudaMalloc(&nb, (size_t)cap * sizeof(BlockDesc)) != cudaSuccess || cudaMalloc(&nc, (size_t)cap * 4) != cudaSuccess)
      return fail(e, NGSQ_E_NOMEM, "cudaMalloc block tables (%u blocks)", cap);
    if (first) {
      CU(cudaMemcpy(nb, e->d_blocks_all, (size_t)first * sizeof(BlockDesc), cudaMemcpyDeviceToDevice));
      CU(cudaMemcpy(nc, e->d_crc_all, (size_t)first * 4, cudaMemcpyDeviceToDevice));
    }
    if (e->d_blocks_all) cudaFree(e->d_blocks_all);
    if (e->d_crc_all) cudaFree(e->d_crc_all);
    e->d_blocks_all = nb; e->d_crc_all = nc; e->blocks_all_cap = cap;
  }
  const uint32_t n = end - first;
  BlockDesc* hb = (BlockDesc*)pin_alloc(e, (size_t)n * sizeof(BlockDesc));
  uint32_t* hc = (uint32_t*)pin_alloc(e, (size_t)n * 4);
  if (!hb || !hc) return fail(e, NGSQ_E_NOMEM, "cudaHostAlloc block tables (%u blocks)", n);
  memcpy(hb, e->h_blocks.data() + first, (size_t)n * sizeof(BlockDesc));
  memcpy(hc, e->h_crc.data() + first, (size_t)n * 4);
  CU(cudaMemcpyAsync(e->d_blocks_all + first, hb, (size_t)n * sizeof(BlockDesc), cudaMemcpyHostToDevice, e->s_copy));
  CU(cudaMemcpyAsync(e->d_crc_all + first, hc, (size_t)n * 4, cudaMemcpyHostToDevice, e->s_copy));
  return NGSQ_OK;
}

// first block with file offset >= co among the current file's blocks [file_b0, n)
uint32_t block_lower_bound(const ngsq_engine* e, uint32_t n, uint64_t co) {
  uint32_t lo = e->file_b0, hi = n;
  while (lo < hi) {
    const uint32_t mid = lo + (hi - lo) / 2;
    if (e->h_blocks[mid].coff < co) lo = mid + 1; else hi = mid;
  }
  return lo;
}

// Resolves the shard's virtual offsets against the blocks submitted so far ([0, n)).  A coffset that names an empty
// (skipped) block resolves to the start of the next real block.
int resolve_range(ngsq_engine* e, uint32_t n) {
  if (!e->start_resolved) {
    const uint64_t co = e->first_voff >> 16;
    uint32_t uo = (uint32_t)(e->first_voff & 0xFFFF);
    const uint32_t b = block_lower_bound(e, n, co);
    if (b < n) {
      if (e->h_blocks[b].coff != co) {
        if (uo) return fail(e, NGSQ_E_ARG, "virtual offset %llu does not address a submitted block", (unsigned long long)e->first_voff);
      } else if (uo > e->h_blocks[b].isize) return fail(e, NGSQ_E_ARG, "virtual offset %llu: uoffset beyond block", (unsigned long long)e->first_voff);
      e->start_block = b; e->start_uo = uo; e->start_resolved = true;
    }
  }
  if (e->end_voff && !e->end_resolved) {
    const uint64_t co = e->end_voff >> 16;
    uint32_t uo = (uint32_t)(e->end_voff & 0xFFFF);
    const uint32_t b = block_lower_bound(e, n, co);
    if (b < n) {
      if (e->h_blocks[b].coff != co) {
        if (uo) return fail(e, NGSQ_E_ARG, "virtual offset %llu does not address a submitted block", (unsigned long long)e->end_voff);
      } else if (uo > e->h_blocks[b].isize) return fail(e, NGSQ_E_ARG, "virtual offset %llu: uoffset beyond block", (unsigned long long)e->end_voff);
      e->end_block = b; e->end_uo = uo; e->end_resolved = true;
    }
  }
  return NGSQ_OK;
}

// K2: lane-per-block Huffman decode, then warp-per-block LZ77 resolve (inflate2.cuh)
int launch_inflate(ngsq_engine* e, const BlockDesc* blocks, uint32_t n, uint8_t* out, uint32_t* queue, uint32_t* status,
                   uint32_t* bitmap, cudaStream_t s, cudaEvent_t ev_decode_from = nullptr, cudaEvent_t ev_decoded = nullptr) {
  if (!n) return NGSQ_OK;
  CU(cudaMemsetAsync(bitmap, 0, (size_t)n * kBitmapWords * 4, s));
  CU(cudaMemsetAsync(status, 0, (size_t)n * 4, s));
  CU(cudaMemsetAsync(queue, 0, 4, s));
  // one CTA per SM as soon as there is a batch of 32 blocks for each (the kernel interleaves batches over the CTAs)
  uint32_t grid = std::min<uint32_t>((n + 31) / 32, (uint32_t)e->n_sm);
  if (ev_decode_from) CU(cudaEventRecord(ev_decode_from, s));
  inflate_decode_kernel<<<grid, kDecThreads, kDecSmem, s>>>(out, blocks, n, queue, status, bitmap);
  CU(cudaGetLastError());
  if (ev_decoded) CU(cudaEventRecord(ev_decoded, s));
  // full occupancy (8 CTAs x 8 warps per SM): measured 39 ms / 40 M records vs 47 / 56 / 79 ms with 4 / 3 / 2 CTAs per SM —
  // latency hiding beats keeping the blocks in flight L2-resident.  One block per warp, no grid-stride loop: the facet
  // kernels of the previous wave share the SMs with this kernel (scan stream), and CTAs that start late must not carry
  // a fixed share of the blocks.
  uint32_t rgrid = (n + kResWarps - 1) / kResWarps;
  inflate_resolve_kernel<<<rgrid, kResThreads, 0, s>>>(out, blocks, n, bitmap, status);
  CU(cudaGetLastError());
  return NGSQ_OK;
}

// NGSQ_F_INDEX: copies the run table of indexed wave j to pinned host memory once its kernel is done, on stream `s` (ahead of
// the kernel of wave j + 2, which reuses the table).  Waits for wave j's index kernel, which by then runs beside the
// inflate of the wave after it.
int ix_drain(ngsq_engine* e, uint32_t j, cudaStream_t s) {
  auto& w = e->ix_waves[j];
  if (w.drained) return NGSQ_OK;
  CU(cudaEventSynchronize(w.done));
  w.drained = true;
  const uint64_t n = std::min<uint64_t>(e->h_ix_probe[j & 1], e->ix_runs_cap);  // more tickets than room: the kernel flagged it
  if (!n) return NGSQ_OK;
  IndexRun* h = (IndexRun*)pin_alloc(e, n * sizeof(IndexRun));
  if (!h) return fail(e, NGSQ_E_NOMEM, "cudaHostAlloc index runs (%llu)", (unsigned long long)n);
  CU(cudaMemcpyAsync(h, e->d_ix_runs[j & 1], n * sizeof(IndexRun), cudaMemcpyDeviceToHost, s));
  e->ix_drained.push_back({h, n});
  return NGSQ_OK;
}

// Device buffers of one wave of n blocks / `bytes` inflated bytes in slot `s`.  Growing a buffer waits for the work in
// flight (only the first waves of a run ever grow anything; reserve_* avoids even that).
int ensure_wave_buffers(ngsq_engine* e, int s, uint32_t n, uint64_t bytes) {
  bool synced = false;
  auto quiesce = [&]() -> int {
    if (synced) return NGSQ_OK;
    CU(cudaStreamSynchronize(e->s_comp));
    CU(cudaStreamSynchronize(e->s_scan));
    CU(cudaStreamSynchronize(e->s_aux));
    synced = true;
    return NGSQ_OK;
  };
  int rc;
  if (bytes > e->slot_cap[s]) {
    if ((rc = quiesce())) return rc;
    // with a reserve hint every slot is sized once for a full wave; otherwise for what the wave needs, with slack
    size_t want = bytes + bytes / 8;
    const uint64_t full = (uint64_t)launch_quantum(e) * 65536;
    if (e->cfg.reserve_inflated) want = (size_t)std::max<uint64_t>(bytes, std::min<uint64_t>(e->cfg.reserve_inflated, full));
    if ((rc = fresh(e, e->d_slot[s], (size_t)e->headroom + want + 512, "inflated slot"))) return rc;
    e->slot_cap[s] = want;
  }
  if (n > e->scan_cap) {
    if ((rc = quiesce())) return rc;
    const uint32_t cap = std::max<uint32_t>(n + n / 8, std::min<uint32_t>(launch_quantum(e), std::max<uint32_t>(e->cfg.reserve_blocks, 64u)));
    if ((rc = fresh(e, e->d_wstatus[0], cap, "status"))) return rc;
    if ((rc = fresh(e, e->d_wstatus[1], cap, "status"))) return rc;
    if ((rc = fresh(e, e->d_first, cap, "scan tables"))) return rc;
    if ((rc = fresh(e, e->d_landed, cap, "scan tables"))) return rc;
    if ((rc = fresh(e, e->d_count, (size_t)cap + 1, "scan tables"))) return rc;
    if ((rc = fresh(e, e->d_base, (size_t)cap + 1, "scan tables"))) return rc;
    e->scan_cap = cap;
  }
  if (n > e->bitmap_cap) {
    if ((rc = quiesce())) return rc;
    const size_t cap = std::max<size_t>(n, e->scan_cap);
    if ((rc = fresh(e, e->d_bitmap, cap * kBitmapWords, "match bitmap"))) return rc;
    e->bitmap_cap = cap;
  }
  const uint64_t need_rec = (e->headroom + std::max<uint64_t>(e->slot_cap[0], e->slot_cap[1])) / 36 + 2;
  if (need_rec > e->rec_cap) {
    if ((rc = quiesce())) return rc;
    if ((rc = fresh(e, e->d_rec, need_rec, "record table"))) return rc;
    e->rec_cap = need_rec;
  }
  // a run starts at a record: the run tables are sized like the record table (the runs of earlier waves are drained first)
  if (ix_on(e) && need_rec > e->ix_runs_cap) {
    if ((rc = quiesce())) return rc;
    for (uint32_t j = 0; j < e->ix_waves.size(); ++j)
      if ((rc = ix_drain(e, j, e->s_scan))) return rc;
    CU(cudaStreamSynchronize(e->s_scan));
    if ((rc = fresh(e, e->d_ix_runs[0], need_rec, "index run table"))) return rc;
    if ((rc = fresh(e, e->d_ix_runs[1], need_rec, "index run table"))) return rc;
    e->ix_runs_cap = need_rec;
  }
  // a read with more than kQualSmemPositions bases takes more than 260 bytes
  const uint64_t need_long = (e->headroom + std::max<uint64_t>(e->slot_cap[0], e->slot_cap[1])) / 260 + 2;
  if ((e->cfg.flags & NGSQ_F_RECORD_FACETS) && need_long > e->long_cap) {
    if ((rc = quiesce())) return rc;
    if ((rc = fresh(e, e->d_long, need_long, "long-read list"))) return rc;
    e->long_cap = need_long;
  }
  if (rg_on(e) && need_rec > e->rg_cap) {
    if ((rc = quiesce())) return rc;
    if ((rc = fresh(e, e->d_rg_of, need_rec, "read-group tags"))) return rc;
    if ((rc = fresh(e, e->d_rg_order, need_rec + 32ull * (e->rg_n + 1), "read-group buckets"))) return rc;
    e->rg_cap = need_rec;
  }
  if ((e->cfg.flags & (NGSQ_F_COVERAGE | NGSQ_F_EDITS)) && e->cfg.max_records && need_rec > e->mark_cap) {
    if ((rc = quiesce())) return rc;
    if ((rc = fresh(e, e->d_mark, need_rec, "record marks"))) return rc;
    e->mark_cap = need_rec;
  }
  return NGSQ_OK;
}

int new_wave_events(ngsq_engine* e, ngsq_engine::Wave& w) {
  for (cudaEvent_t* x : {&w.begin, &w.decoded_from, &w.decoded, &w.resolved, &w.scan_begin, &w.begun, &w.scan_end, &w.facets_end, &w.crc_begin, &w.crc_end}) CU(cudaEventCreate(x));
  return NGSQ_OK;
}

// CRC32 of a wave's blocks against their trailers (what noodles-bgzf checks per block), on its own stream.  The kernel's
// shared-memory tables cannot share an SM with the decoder, and a CRC kernel that reached the SMs first would hold the
// next wave's decode back; so it is enqueued behind the START of the next wave's decode (`after`; lowest stream
// priority) and fills the SMs as the decoder leaves them, beside that wave's resolve.  The last wave's follows it at once.
int launch_crc(ngsq_engine* e, ngsq_engine::Wave& w, cudaEvent_t after) {
  if (w.crc_launched) return NGSQ_OK;
  w.crc_launched = true;
  CU(cudaStreamWaitEvent(e->s_aux, w.resolved, 0));
  if (after) CU(cudaStreamWaitEvent(e->s_aux, after, 0));
  CU(cudaEventRecord(w.crc_begin, e->s_aux));
  if (e->cfg.flags & NGSQ_F_VERIFY_CRC) {
    const uint32_t n = w.b1 - w.b0;
    const uint32_t grid = (n + kCrcThreads / 32 - 1) / (kCrcThreads / 32);  // one block per warp: late CTAs carry no fixed share
    crc32_kernel<<<grid, kCrcThreads, kCrcSmem, e->s_aux>>>(w.out, e->d_blocks_all + w.b0, e->d_crc_all + w.b0, n, e->d_crc_tables, &e->d_state->crc_bad);
    CU(cudaGetLastError());
    e->other_launches++;
  }
  CU(cudaEventRecord(w.crc_end, e->s_aux));
  return NGSQ_OK;
}

// One wave: blocks [b0, b1) -> inflate -> CRC (own stream) -> record scan -> facet kernels.  Nothing here waits for the GPU
// (except when a buffer has to grow).
int launch_wave(ngsq_engine* e, uint32_t b0, uint32_t b1, bool final_wave) {
  const uint32_t n = b1 - b0;
  if (!n) return NGSQ_OK;
  if (!e->range_set) return fail(e, NGSQ_E_ARG, "ngsq_set_range was not called");
  int rc = resolve_range(e, b1);
  if (rc) return rc;
  const uint32_t wi = (uint32_t)e->waves.size();
  const int s = (int)(wi & 1);
  if (e->trace) {
    timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts);
    const double now = ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
    if (!wi) e->host_t0 = now;
    e->host_ms.push_back(now - e->host_t0);
  }
  // Two kernel streams: inflate (decode + resolve) on s_comp, record scan + facet kernels on s_scan, so that the scan of
  // wave k runs beside the decode of wave k + 1 (the decoder owns the SMs' shared memory but leaves thread and register
  // room) and its facet kernels beside the resolve of wave k + 1.
  cudaStream_t st = e->s_comp;
  const uint64_t out0 = e->h_blocks[b0].out_off;
  const uint64_t bytes = e->h_blocks[b1 - 1].out_off + e->h_blocks[b1 - 1].isize - out0;
  // slot s and the status table of this parity were last used by wave wi - 2: its CRC kernel (own stream), its scan and
  // facet kernels, and the copy of its open record into wave wi - 1's headroom (`begun` of wave wi - 1 is recorded
  // behind all of these on the in-order scan stream) must be done with them
  if (wi >= 2) CU(cudaStreamWaitEvent(st, e->waves[wi - 2].crc_end, 0));
  if (wi >= 1) CU(cudaStreamWaitEvent(st, e->waves[wi - 1].begun, 0));
  if ((rc = ensure_wave_buffers(e, s, n, bytes))) return rc;
  // the compressed bytes of the wave: wait for the copy of the last chunk it reads
  for (const auto& c : e->chunks)
    if (c.blocks_end >= b1) { CU(cudaStreamWaitEvent(st, c.copied, 0)); break; }
  ngsq_engine::Wave w{};
  if ((rc = new_wave_events(e, w))) return rc;
  w.b1 = b1;
  uint8_t* slot = e->d_slot[s];
  // descriptors carry offsets in the whole inflated stream; the wave's first block lands right behind the headroom
  uint8_t* out = slot + e->headroom - out0;
  const BlockDesc* wblocks = e->d_blocks_all + b0;
  CU(cudaEventRecord(w.begin, st));
  uint32_t* wstatus = e->d_wstatus[s];
  rc = launch_inflate(e, wblocks, n, out, e->d_queue, wstatus, e->d_bitmap, st, w.decoded_from, w.decoded);
  if (rc) return rc;
  e->other_launches += 1;  // resolve kernel (the decode kernel is counted as the inflate launch)
  CU(cudaEventRecord(w.resolved, st));
  // the previous wave's CRC kernel becomes eligible when this wave's decode starts (see launch_crc)
  w.b0 = b0; w.out = out; w.crc_launched = false;
  const bool serial = e->cfg.flags & NGSQ_F_SERIAL_STAGES;  // measurement aid: one kernel stream, CRC beside this wave's scan
  if (serial) { if ((rc = launch_crc(e, w, nullptr))) return rc; }
  else if (wi >= 1 && (rc = launch_crc(e, e->waves[wi - 1], w.decoded_from))) return rc;

  // ---- K3: which part of the wave does the shard own?
  const bool before_start = !e->start_resolved || e->start_block >= b1;
  const bool after_end = e->end_resolved && e->end_block < b0;
  w.scanned = !before_start && !after_end;
  st = serial ? e->s_comp : e->s_scan;
  CU(cudaStreamWaitEvent(st, w.resolved, 0));
  CU(cudaEventRecord(w.scan_begin, st));
  if (!w.scanned) {
    status_fold_kernel<<<(n + 255) / 256, 256, 0, st>>>(wstatus, n, b0, e->d_state);
    CU(cudaGetLastError());
    e->other_launches++;
    CU(cudaEventRecord(w.begun, st));
    CU(cudaEventRecord(w.scan_end, st));
    CU(cudaEventRecord(w.facets_end, st));
    e->waves.push_back(w);
    e->stats.inflate_launches++;
    return NGSQ_OK;
  }
  WaveParams W{};
  W.d = slot; W.out0 = out0; W.blocks = wblocks; W.status = wstatus; W.n_blocks = n; W.first_global = b0; W.headroom = e->headroom;
  W.first_wave = e->start_block >= b0 ? 1u : 0u;
  W.final_wave = final_wave ? 1u : 0u;
  W.n_ref = (int32_t)e->n_ref;
  W.wave_end = (uint64_t)e->headroom + bytes;
  W.start_off = W.first_wave ? (uint64_t)e->headroom + (e->h_blocks[e->start_block].out_off - out0) + e->start_uo : 0;
  W.end_off = ~0ull;
  if (e->end_resolved && e->end_block < b1) W.end_off = (uint64_t)e->headroom + (e->h_blocks[e->end_block].out_off - out0) + e->end_uo;
  W.rec_cap = e->rec_cap;
  W.st = e->d_state; W.first = e->d_first; W.landed = e->d_landed; W.count = e->d_count; W.base = e->d_base; W.rec = e->d_rec;
  // the previous scanned wave sits in the other slot (waves outside the range carry nothing)
  const uint8_t* prev = (wi && e->waves[wi - 1].scanned) ? e->d_slot[s ^ 1] : nullptr;
  CU(cudaMemsetAsync(e->d_landed, 0, (size_t)n * 4, st));
  // single-CTA kernels of the scan chain use 256 threads: beside a resident decoder CTA (576 threads x 96 registers, all
  // but 4 KB of the shared memory) an SM has room for about 10 K registers
  wave_begin_kernel<<<1, 256, 0, st>>>(e->d_state, slot, prev, e->headroom, W.first_wave);
  CU(cudaEventRecord(w.begun, st));  // the other slot is free for the next wave's inflate
  find_first_kernel<<<(n * 32 + 255) / 256, 256, 0, st>>>(W);
  const uint32_t wg = (n + 1 + 127) / 128;
  walk_kernel<false, false><<<wg, 128, 0, st>>>(W);
  check_landed_kernel<false><<<(n + 255) / 256, 256, 0, st>>>(W);
  chain_fix_kernel<<<1, 256, 0, st>>>(W);
  walk_kernel<false, true><<<wg, 128, 0, st>>>(W);
  check_landed_kernel<true><<<(n + 255) / 256, 256, 0, st>>>(W);
  scan_counts_kernel<<<1, 256, 0, st>>>(W);
  walk_kernel<true, false><<<wg, 128, 0, st>>>(W);
  CU(cudaGetLastError());
  e->other_launches += 9;
  CU(cudaMemcpyAsync(e->h_prog + 2 * (wi % kProgSlots), &e->d_state->rec_base, 16, cudaMemcpyDeviceToHost, st));
  CU(cudaEventRecord(w.scan_end, st));

  // ---- K4-K8 (+ K11, K12)
  const bool cov_n = (e->cfg.flags & NGSQ_F_COVERAGE) && e->cfg.max_records;
  if (e->cfg.flags & (NGSQ_F_RECORD_FACETS | NGSQ_F_COVERAGE)) {
    FacetParams P{};
    P.d = slot; P.rec = e->d_rec; P.st = e->d_state; P.st_w = e->d_state; P.blocks = wblocks; P.headroom = e->headroom; P.out0 = out0;
    P.cov_scatter = cov_n ? 0u : 1u;
    P.max_records = e->cfg.max_records; P.gc_seed = e->cfg.gc_seed; P.n_ref = (int32_t)e->n_ref; P.flags = e->cfg.flags;
    P.ref_len = e->d_ref_len; P.cov_enabled = e->d_cov_enabled; P.diff_base = e->d_diff_base; P.diff = e->d_diff; P.cov_slot = e->d_cov_slot;
    P.tile_off = e->d_tile_off; P.tile_sum = e->d_tile_sum;
    P.res = e->d_res; P.qual = e->d_res + e->qual_off;
    P.qpos_smem = kQualSmemPositions;
    P.qpos_cap = e->qpos_cap;
    P.long_list = e->d_long; P.long_cap = (uint32_t)std::min<uint64_t>(e->long_cap, 0xFFFFFFFFu);
    // persistent grid sized for the bound "a record is at least 36 bytes": the record count stays on the device
    const uint64_t want = (bytes / 36 + 2 + kFacetThreads - 1) / kFacetThreads;
    const uint32_t grid = (uint32_t)std::min<uint64_t>(want, (uint64_t)e->n_sm * e->facet_occ);
    facets_kernel<<<grid, kFacetThreads, e->facet_smem, st>>>(P);
    CU(cudaGetLastError());
    e->other_launches++;
    if (e->cfg.flags & NGSQ_F_RECORD_FACETS) {
      // quality positions beyond the shared-memory tables; both kernels return at once on a wave without such reads
      QualTileParams T{};
      T.d = slot; T.list = e->d_long; T.long_cap = P.long_cap; T.st = e->d_state; T.qual = P.qual; T.res = e->d_res;
      T.qpos_smem = kQualSmemPositions; T.qpos_cap = e->qpos_cap;
      qual_tiles_kernel<<<e->n_sm * 2, kTileThreads, kTileSmem, st>>>(T);
      qual_verdict_kernel<<<e->n_sm, 256, 0, st>>>(T);
      CU(cudaGetLastError());
      e->other_launches += 2;
    }
    if (rg_on(e)) {
      // the four record facets per read group: tag, bucket, tally (read_groups.cuh)
      ReadGroupParams G{};
      G.d = slot; G.rec = e->d_rec; G.st = e->d_state; G.blocks = wblocks; G.headroom = e->headroom; G.out0 = out0;
      G.max_records = e->cfg.max_records; G.gc_seed = e->cfg.gc_seed; G.n_ref = (int32_t)e->n_ref;
      G.n_groups = e->rg_n; G.ids = e->d_rg_ids; G.id_off = e->d_rg_id_off; G.table = e->d_rg_table; G.mask = e->rg_mask;
      G.grp = e->d_rg_of; G.count = e->d_rg_count; G.cursor = e->d_rg_cursor; G.order = e->d_rg_order; G.total = e->d_rg_total;
      const uint64_t ng = (uint64_t)e->rg_n + 1;
      G.sums = e->d_grp; G.qlen = e->d_grp + ng * kGroupSums; G.qual = e->d_grp + ng * (kGroupSums + 1); G.rows = e->grp_rows;
      G.res = e->d_res;
      const uint32_t tgrid = (uint32_t)std::min<uint64_t>((bytes / 36 + 2 + kRgThreads - 1) / kRgThreads, (uint64_t)e->n_sm * 8);
      rg_tag_kernel<<<tgrid, kRgThreads, 0, st>>>(G);
      rg_scan_kernel<<<1, kRgScanThreads, 0, st>>>(G);
      rg_scatter_kernel<<<tgrid, kRgThreads, 0, st>>>(G);
      rg_facets_kernel<<<(uint32_t)e->n_sm * e->rg_occ, kFacetThreads, e->rg_smem, st>>>(G);
      CU(cudaGetLastError());
      e->other_launches += 4;
    }
  }
  // `-n`: which records the second pass processes (one counter over all sequences) — Coverage and Edits share the marks
  const bool pass2_n = (e->cfg.flags & (NGSQ_F_COVERAGE | NGSQ_F_EDITS)) && e->cfg.max_records;
  if (pass2_n) {
    CovNParams C{};
    C.d = slot; C.rec = e->d_rec; C.st = e->d_state; C.max_records = e->cfg.max_records; C.n_ref = (int32_t)e->n_ref;
    C.ref_len = e->d_ref_len; C.cov_enabled = e->d_cov_enabled; C.diff_base = e->d_diff_base; C.diff = e->d_diff; C.cov_slot = e->d_cov_slot;
    C.tile_off = e->d_tile_off; C.tile_sum = e->d_tile_sum;
    C.res = e->d_res; C.mark = e->d_mark;
    const uint32_t grid = (uint32_t)std::min<uint64_t>((bytes / 36 + 2 + 255) / 256, (uint64_t)e->n_sm * 8);
    cov_n_mark_kernel<<<grid, 256, 0, st>>>(C);
    cov_n_rank_kernel<<<1, 1024, 0, st>>>(C);
    if (cov_n) cov_n_apply_kernel<<<grid, 256, 0, st>>>(C);
    CU(cudaGetLastError());
    e->other_launches += cov_n ? 3 : 2;
  }
  const uint32_t rgrid = (uint32_t)std::min<uint64_t>((bytes / 36 + 2 + 255) / 256, (uint64_t)e->n_sm * 8);
  if ((e->cfg.flags & NGSQ_F_EDITS) && e->d_ed_res && e->ed_contigs.size() == e->n_ref) {
    // K11: per-record edit counts and per-position ref / alt counters (the VAF histogram follows in ngsq_finish)
    EditsParams EP{};
    EP.d = slot; EP.rec = e->d_rec; EP.st = e->d_state; EP.n_ref = (int32_t)e->n_ref;
    EP.contigs = e->d_ed_contigs; EP.refs = e->d_ed_refs; EP.alts = e->d_ed_alts; EP.res = e->d_ed_res;
    EP.mark = pass2_n ? e->d_mark : nullptr;
    edits_kernel<<<rgrid, 256, 0, st>>>(EP);
    CU(cudaGetLastError());
    e->other_launches++;
  }
  if ((e->cfg.flags & NGSQ_F_FEATURES) && e->d_ft_res && e->ft_model_set && e->ft_contigs.size() == e->n_ref) {
    // K12: per-record overlap counts against the gene model
    FeatureParams FP{};
    FP.d = slot; FP.rec = e->d_rec; FP.st = e->d_state; FP.max_records = e->cfg.max_records; FP.n_ref = (int32_t)e->n_ref;
    FP.contigs = e->d_ft_contigs; FP.res = e->d_ft_res;
    memcpy(FP.slot_class, e->ft_slot_class, 8);
    features_kernel<<<rgrid, 256, 0, st>>>(FP);
    CU(cudaGetLastError());
    e->other_launches++;
  }
  if (ix_on(e)) {
    // K13: keys, runs, order check, counters and linear index of the wave's records
    const uint32_t j = (uint32_t)e->ix_waves.size(), par = j & 1;
    if (j >= 2 && (rc = ix_drain(e, j - 2, st))) return rc;
    CU(cudaMemsetAsync(&e->d_ix->n_runs[par], 0, 8, st));
    IndexParams X{};
    X.d = slot; X.rec = e->d_rec; X.st = e->d_state; X.blocks = wblocks; X.headroom = e->headroom; X.par = par; X.out0 = out0;
    X.n_ref = (int32_t)e->n_ref; X.S = e->d_ix; X.runs = e->d_ix_runs[par]; X.runs_cap = e->ix_runs_cap;
    X.ovf = e->d_ix_ovf; X.ovf_cap = kIndexOverflowCap;
    X.win_base = e->d_ix_win_base; X.win_n = e->d_ix_win_n; X.win = e->d_ix_win; X.max_win = e->d_ix_maxw; X.counts = e->d_ix_counts;
    X.part = (e->cfg.flags & NGSQ_F_INDEX_PART) ? 1u : 0u;
    X.min_shift = e->ix_min_shift; X.depth = e->ix_depth;
    const uint32_t per_cta = 31 * (kIndexThreads / 32);
    const uint32_t xgrid = (uint32_t)std::min<uint64_t>((bytes / 36 + 2 + per_cta - 1) / per_cta, (uint64_t)e->n_sm * 8);
    if (ix_csi(e)) index_kernel<true><<<xgrid, kIndexThreads, 0, st>>>(X);
    else index_kernel<false><<<xgrid, kIndexThreads, 0, st>>>(X);
    CU(cudaGetLastError());
    e->other_launches++;
    CU(cudaMemcpyAsync(e->h_ix_probe + par, &e->d_ix->n_runs[par], 8, cudaMemcpyDeviceToHost, st));
    ngsq_engine::IxWave xw{nullptr, false};
    CU(cudaEventCreateWithFlags(&xw.done, cudaEventDisableTiming));
    e->ix_waves.push_back(xw);
    CU(cudaEventRecord(xw.done, st));
  }
  CU(cudaEventRecord(w.facets_end, st));
  e->waves.push_back(w);
  e->stats.inflate_launches++;
  return NGSQ_OK;
}

// Hands blocks [launched, upto) to the kernels, one wave per `quantum` blocks.
int launch_pending(ngsq_engine* e, uint32_t upto, bool final_wave) {
  const uint32_t quantum = launch_quantum(e);
  while (e->launched < upto) {
    const uint32_t b1 = std::min(upto, e->launched + quantum);
    int rc = launch_wave(e, e->launched, b1, final_wave && b1 == upto);
    if (rc) return rc;
    e->launched = b1;
  }
  return NGSQ_OK;
}

// A compressed segment is free again once the wave that reads its last block has been decoded.
bool seg_retired(ngsq_engine* e, const ngsq_engine::CompSeg& sg, bool wait) {
  if (!sg.blocks_end) return true;  // holds no blocks
  if (sg.blocks_end > e->launched) return false;
  for (const auto& w : e->waves)
    if (w.b1 >= sg.blocks_end) {
      if (wait) return cudaEventSynchronize(w.decoded) == cudaSuccess;
      return cudaEventQuery(w.decoded) == cudaSuccess;
    }
  return false;
}

// Device space for `nbytes` of compressed input: the open segment, a retired one, a new one while the ring may grow;
// otherwise the caller waits for the oldest wave (back-pressure on the submitting thread).
int acquire_comp(ngsq_engine* e, size_t nbytes, uint8_t** dst) {
  const size_t need = (nbytes + 15) & ~size_t(15);
  if (!e->comp_segs.empty()) {
    auto& b = e->comp_segs.back();
    if (b.used + need <= b.cap) { *dst = b.ptr + b.used; b.used += need; return NGSQ_OK; }
  }
  auto reuse = [&](size_t i) {
    ngsq_engine::CompSeg take = e->comp_segs[i];
    e->comp_segs.erase(e->comp_segs.begin() + i);
    take.used = need; take.blocks_end = 0;
    e->comp_segs.push_back(take);
    *dst = take.ptr;
  };
  for (size_t i = 0; i < e->comp_segs.size(); ++i)
    if (e->comp_segs[i].cap >= need && seg_retired(e, e->comp_segs[i], false)) { reuse(i); return NGSQ_OK; }
  const size_t limit = e->cfg.comp_ring_bytes ? (size_t)e->cfg.comp_ring_bytes : kDefaultCompRing;
  // segments of a quarter of the ring (at most 256 MB): one being filled, the others under the decoders
  const size_t cap = std::max<size_t>(need, std::min<size_t>((size_t)256 << 20, std::max<size_t>(limit / 4, (size_t)1 << 20)));
  if (!e->comp_segs.empty() && e->comp_total + cap > limit) {
    // the ring is full: hand every block that is still waiting to a (smaller) wave, then wait for the oldest segment
    int rc = launch_pending(e, (uint32_t)e->h_blocks.size(), false);
    if (rc) return rc;
    for (size_t i = 0; i < e->comp_segs.size(); ++i)
      if (e->comp_segs[i].cap >= need && seg_retired(e, e->comp_segs[i], true)) { reuse(i); return NGSQ_OK; }
    // no segment is large enough for this chunk: grow past the limit
  }
  uint8_t* p = nullptr;
  cudaError_t r2 = cudaMalloc(&p, cap + 512);
  if (r2 != cudaSuccess) return fail(e, NGSQ_E_NOMEM, "cudaMalloc compressed segment (%zu bytes): %s", cap, cudaGetErrorString(r2));
  e->comp_segs.push_back({p, cap, need, 0});
  e->comp_total += cap;
  *dst = p;
  return NGSQ_OK;
}

// K13 on the host, the part a BAI and a CSI share: runs -> chunks per (reference, bin), merged where they touch, bins in order
// of first use; the per-window minimum offsets, untouched windows filled with the previous window's value (0 before the
// first touched one).  For the state H (one engine's, or the join of several parts').  Sorts H.runs.
struct IxRef {
  std::vector<std::pair<uint32_t, std::vector<std::pair<uint64_t, uint64_t>>>> bins;  // in order of first use
  uint64_t beg = 0, end = 0;
  bool any = false;
  std::vector<uint64_t> win;  // windows 0 ..= the last touched one, filled
};
size_t ix_collect(IxHost& H, uint32_t nr, uint32_t n_bins, const std::vector<uint64_t>& win_base, const std::vector<uint32_t>& win_n,
                  std::vector<IxRef>& refs) {
  std::vector<IndexRun>& runs = H.runs;
  // runs were ticketed in any order; each starts at a distinct record, and run r ends where run r + 1 starts
  std::sort(runs.begin(), runs.end(), [](const IndexRun& a, const IndexRun& b) { return a.voff < b.voff; });
  refs.assign(nr, IxRef{});
  const uint64_t data_end = H.data_end;
  // the runs of one reference are consecutive (sorted input): one bin -> slot table, cleared when the reference changes
  std::vector<int32_t> slot_of(n_bins + 1, -1);
  uint32_t cur = kIxUnplacedRef;
  size_t chunks = 0;
  for (size_t i = 0; i < runs.size(); ++i) {
    const IndexRun& u = runs[i];
    if (u.ref == kIxUnplacedRef) continue;
    const uint64_t end = i + 1 < runs.size() ? runs[i + 1].voff : data_end;
    IxRef& R = refs[u.ref];
    if (u.ref != cur) {
      if (cur != kIxUnplacedRef) for (auto& bn : refs[cur].bins) slot_of[bn.first] = -1;
      cur = u.ref;
    }
    if (!R.any) { R.any = true; R.beg = u.voff; }
    R.end = end;
    int32_t& sl = slot_of[u.bin];
    if (sl < 0) { sl = (int32_t)R.bins.size(); R.bins.push_back({u.bin, {}}); }
    auto& ch = R.bins[sl].second;
    // contiguous with the bin's last chunk (also a run that a cut between two parts split in two)
    if (!ch.empty() && ch.back().second == u.voff) ch.back().second = end;
    else { ch.push_back({u.voff, end}); ++chunks; }
  }
  for (uint32_t c = 0; c < nr; ++c) {
    IxRef& R = refs[c];
    if (!R.any) continue;
    const uint32_t n_intv = H.maxw[c] + 1;
    std::vector<uint64_t>& lin = R.win;
    lin.assign(n_intv, ~0ull);
    const uint32_t in_table = std::min(n_intv, win_n[c]);
    for (uint32_t w = 0; w < in_table; ++w) lin[w] = H.win[win_base[c] + w];
    for (const IndexOvf& o : H.ovf)
      if (o.ref == c)
        for (uint32_t w = o.lo; w <= o.hi && w < n_intv; ++w) lin[w] = std::min(lin[w], o.voff);
    uint64_t last = 0;
    for (uint32_t w = 0; w < n_intv; ++w) {
      if (lin[w] == ~0ull) lin[w] = last; else last = lin[w];
    }
  }
  return chunks;
}

// The .bai bytes: per reference its bins and chunks, the pseudo-bin 37450 and the linear index; n_no_coor.
void assemble_bai(IxHost& H, uint32_t nr, const std::vector<uint64_t>& win_base, const std::vector<uint32_t>& win_n, std::vector<uint8_t>& b) {
  std::vector<IxRef> refs;
  const size_t chunks = ix_collect(H, nr, kIxMetaBin - 1, win_base, win_n, refs);
  size_t wins = 0;
  for (const IxRef& R : refs) wins += R.win.size();
  b.clear();
  b.reserve(16 + (size_t)nr * 64 + chunks * 16 + wins * 8);
  auto p32 = [&](uint32_t v) { uint8_t t[4]; memcpy(t, &v, 4); b.insert(b.end(), t, t + 4); };
  auto p64 = [&](uint64_t v) { uint8_t t[8]; memcpy(t, &v, 8); b.insert(b.end(), t, t + 8); };
  b.insert(b.end(), {'B', 'A', 'I', 1});
  p32(nr);
  for (uint32_t c = 0; c < nr; ++c) {
    const IxRef& R = refs[c];
    if (!R.any) { p32(0); p32(0); continue; }
    p32((uint32_t)R.bins.size() + 1);
    for (auto& bn : R.bins) {
      p32(bn.first);
      p32((uint32_t)bn.second.size());
      for (auto& ck : bn.second) { p64(ck.first); p64(ck.second); }
    }
    p32(kIxMetaBin); p32(2); p64(R.beg); p64(R.end); p64(H.counts[2 * c]); p64(H.counts[2 * c + 1]);
    p32((uint32_t)R.win.size());
    for (uint64_t v : R.win) p64(v);
  }
  p64(H.S.n_no_coor);
}

// The .csi payload (CSIv1, uncompressed): magic, min_shift, depth, l_aux = 0, n_ref; per reference its bins, each with its
// loffset (the filled window minimum at the bin's first leaf window, 0 past the last touched window) and chunks, then the
// pseudo-bin n_bins + 1 with loffset 0; n_no_coor.  No linear index.
void assemble_csi(IxHost& H, uint32_t nr, uint32_t min_shift, uint32_t depth, const std::vector<uint64_t>& win_base,
                  const std::vector<uint32_t>& win_n, std::vector<uint8_t>& b) {
  std::vector<IxRef> refs;
  const uint32_t n_bins = ix_csi_n_bins(depth);
  const size_t chunks = ix_collect(H, nr, n_bins, win_base, win_n, refs);
  size_t bins = 0;
  for (const IxRef& R : refs) bins += R.bins.size();
  b.clear();
  b.reserve(24 + (size_t)nr * 64 + chunks * 16 + bins * 16);
  auto p32 = [&](uint32_t v) { uint8_t t[4]; memcpy(t, &v, 4); b.insert(b.end(), t, t + 4); };
  auto p64 = [&](uint64_t v) { uint8_t t[8]; memcpy(t, &v, 8); b.insert(b.end(), t, t + 8); };
  b.insert(b.end(), {'C', 'S', 'I', 1});
  p32(min_shift); p32(depth); p32(0); p32(nr);
  for (uint32_t c = 0; c < nr; ++c) {
    const IxRef& R = refs[c];
    if (!R.any) { p32(0); continue; }
    p32((uint32_t)R.bins.size() + 1);
    for (auto& bn : R.bins) {
      const uint64_t bot = ix_csi_bin_bot(bn.first, depth);
      p32(bn.first);
      p64(bot < R.win.size() ? R.win[bot] : 0);
      p32((uint32_t)bn.second.size());
      for (auto& ck : bn.second) { p64(ck.first); p64(ck.second); }
    }
    p32(n_bins + 1); p64(0); p32(2); p64(R.beg); p64(R.end); p64(H.counts[2 * c]); p64(H.counts[2 * c + 1]);
  }
  p64(H.S.n_no_coor);
}

// the index bytes of the state H in the engine's format
void assemble_index(const ngsq_engine* e, IxHost& H, std::vector<uint8_t>& b) {
  if (ix_csi(e)) assemble_csi(H, e->n_ref, e->ix_min_shift, e->ix_depth, e->ix_win_base, e->ix_win_n, b);
  else assemble_bai(H, e->n_ref, e->ix_win_base, e->ix_win_n, b);
}

int fail_unsorted(ngsq_engine* e, uint64_t voff) {
  return fail(e, NGSQ_E_UNSORTED, "the records are not coordinate-sorted: the record at virtual offset %llu (block at file offset %llu, offset %llu) "
              "comes after a record with a larger (reference, position) or an unplaced one; sort the file before indexing it",
              (unsigned long long)voff, (unsigned long long)(voff >> 16), (unsigned long long)(voff & 0xFFFF));
}

// K13 at ngsq_finish: the index state back from the device (the run tables drained so far, the rest now), its error bits;
// then the .bai bytes (NGSQ_F_INDEX) or the part's state for the join (NGSQ_F_INDEX_PART).
int finish_index(ngsq_engine* e) {
  for (uint32_t j = 0; j < e->ix_waves.size(); ++j) {
    int rc = ix_drain(e, j, e->s_comp);
    if (rc) return rc;
  }
  CU(cudaStreamSynchronize(e->s_comp));
  IxHost& H = e->ix;
  H = IxHost{};
  IndexState& S = H.S;
  CU(cudaMemcpy(&S, e->d_ix, sizeof S, cudaMemcpyDeviceToHost));
  if (S.err & kIxBadRecord) return fail(e, NGSQ_E_BAD_RECORD, "malformed BAM record (field overrun, CIGAR op > 8 or reference id out of range)");
  if ((S.err & kIxTooLong) && ix_csi(e))
    return fail(e, NGSQ_E_BAD_RECORD, "a record ends beyond position 2^%u, which a CSI of min_shift %u and depth %u cannot address",
                e->ix_min_shift + 3 * e->ix_depth, e->ix_min_shift, e->ix_depth);
  if (S.err & kIxTooLong) return fail(e, NGSQ_E_BAD_RECORD, "a record ends beyond position 2^29, which a BAI cannot address (CSI can)");
  if (S.err & kIxRunTable) return fail(e, NGSQ_E_CHAIN, "index run table overflow");
  if (S.err & kIxOverflowList)
    return fail(e, NGSQ_E_NOMEM, "more than %llu records reach past the end of their reference sequence", (unsigned long long)kIndexOverflowCap);
  const bool part = e->cfg.flags & NGSQ_F_INDEX_PART;
  if (!part && S.unsorted_voff != ~0ull) return fail_unsorted(e, S.unsorted_voff);
  const uint32_t nr = e->n_ref;
  H.win.resize(e->ix_win_total);
  H.counts.resize((size_t)nr * 2);
  H.maxw.resize(nr);
  if (e->ix_win_total) CU(cudaMemcpy(H.win.data(), e->d_ix_win, e->ix_win_total * 8, cudaMemcpyDeviceToHost));
  if (nr) {
    CU(cudaMemcpy(H.counts.data(), e->d_ix_counts, (size_t)nr * 16, cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(H.maxw.data(), e->d_ix_maxw, (size_t)nr * 4, cudaMemcpyDeviceToHost));
  }
  const size_t n_ovf = std::min<uint64_t>(S.n_ovf, kIndexOverflowCap);
  H.ovf.resize(n_ovf);
  if (n_ovf && ix_csi(e)) CU(cudaMemcpy(H.ovf.data(), e->d_ix_ovf, n_ovf * sizeof(IndexOvf), cudaMemcpyDeviceToHost));
  else if (n_ovf) {
    std::vector<IndexRun> packed(n_ovf);
    CU(cudaMemcpy(packed.data(), e->d_ix_ovf, n_ovf * sizeof(IndexRun), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < n_ovf; ++i) H.ovf[i] = IndexOvf{packed[i].voff, packed[i].ref, packed[i].bin & 0xFFFF, packed[i].bin >> 16, 0};
  }
  for (auto& d : e->ix_drained) H.runs.insert(H.runs.end(), d.first, d.first + d.second);
  H.last_order_key = S.carry[e->ix_waves.size() & 1].order_key;  // the carry the last indexed wave wrote
  H.data_end = e->data_end_coff << 16;
  if (part) { e->ix_part_ok = true; return NGSQ_OK; }
  assemble_index(e, H, e->ix_bytes);
  H = IxHost{};
  return NGSQ_OK;
}

// K9 for contig c: scan of its tile sums, then the streaming resolve into its result slot (both skip an untouched contig)
void launch_cov_resolve(ngsq_engine* e, uint32_t c, cudaStream_t s) {
  uint32_t n = e->ref_len[c] + 1;
  uint32_t n_tiles = (n + kCovTile - 1) / kCovTile;
  const int32_t* df = e->d_diff + e->diff_base[c];
  uint64_t* slot = e->d_res + e->cov_slot[c];
  cov_scan_tiles_kernel<<<1, 1024, 0, s>>>(e->d_tile_sum + e->tile_off[c], e->d_tile, n_tiles, slot + COV_TOUCHED);
  const uint32_t grid = std::min<uint32_t>(n_tiles, e->n_sm * 4);
  cov_resolve_kernel<<<grid, kCovThreads, 0, s>>>(df, n, e->d_tile, n_tiles, slot);
  e->other_launches += 2;
}

// K11 teardown over the per-position counters [off, off + n)
void launch_vaf(ngsq_engine* e, uint64_t off, uint64_t n, cudaStream_t s) {
  const uint32_t vgrid = (uint32_t)std::min<uint64_t>((n + 255) / 256, (uint64_t)e->n_sm * 8);
  edits_vaf_kernel<<<vgrid, 256, 0, s>>>(e->d_ed_refs + off, e->d_ed_alts + off, n, e->d_ed_res);
  e->other_launches += 1;
}

uint32_t cov_tiles(const ngsq_engine* e, uint32_t c) { return (uint32_t)(((uint64_t)e->ref_len[c] + 1 + kCovTile - 1) / kCovTile); }
bool is_split(const ngsq_engine* e, uint32_t c) { return c < e->split_ref.size() && e->split_ref[c]; }
bool edits_loaded(const ngsq_engine* e) { return (e->cfg.flags & NGSQ_F_EDITS) && e->d_ed_res && e->ed_contigs.size() == e->n_ref; }

// Folded into the layout word the ranks agree on: 0 without split references, so that layout stays what it was.
uint64_t split_signature(const ngsq_engine* e) {
  uint64_t h = 0;
  for (uint32_t c = 0; c < e->n_ref; ++c) {
    if (!e->split_ref[c]) continue;
    uint64_t z = h ^ (0x9E3779B97F4A7C15ull * (c + 1ull));
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    h = z ^ (z >> 31);
  }
  return e->n_split ? (h | 1) : 0;
}

// Once every rank's split arrays have been summed into the root's: the root resolves its split references (K9 and the VAF
// pass over their counters; a contig is resolved iff some rank touched it); every other rank zeroes its partials, so that
// per-position reads and later sums of result buffers count each position once.  Enqueued on s.
int merge_split_local(ngsq_engine* e, bool is_root, cudaStream_t s) {
  const bool edits = edits_loaded(e) && e->ed_pos_total;
  for (uint32_t c = 0; c < e->n_ref; ++c) {
    if (!e->split_ref[c]) continue;
    if (is_root) {
      if (e->cov_enabled[c]) launch_cov_resolve(e, c, s);
      if (edits) launch_vaf(e, e->ed_contigs[c].pos_off, (uint64_t)e->ed_contigs[c].hdr_len + 1, s);
    } else {
      if (e->cov_enabled[c]) {
        CU(cudaMemsetAsync(e->d_diff + e->diff_base[c], 0, ((uint64_t)e->ref_len[c] + 2) * 4, s));
        CU(cudaMemsetAsync(e->d_tile_sum + e->tile_off[c], 0, (size_t)cov_tiles(e, c) * 4, s));
        CU(cudaMemsetAsync(e->d_res + e->cov_slot[c] + COV_TOUCHED, 0, 8, s));
      }
      if (edits) {
        const EditsContig& ec = e->ed_contigs[c];
        CU(cudaMemsetAsync(e->d_ed_refs + ec.pos_off, 0, ((uint64_t)ec.hdr_len + 1) * 4, s));
        CU(cudaMemsetAsync(e->d_ed_alts + ec.pos_off, 0, ((uint64_t)ec.hdr_len + 1) * 4, s));
      }
    }
  }
  CU(cudaGetLastError());
  return NGSQ_OK;
}

// Whole BGZF blocks inflated into device memory on s_copy by the engine's inflate kernels (ngsq_inflate_to_host,
// ngsq_find_record); freed with the object.
struct DevInflated {
  uint8_t *in = nullptr, *out = nullptr;
  BlockDesc* blocks = nullptr;
  uint32_t *status = nullptr, *bitmap = nullptr;  // status: one word per block, then the decoder's queue word and 60 spare bytes
  std::vector<BlockDesc> hb;                      // non-empty blocks; coff absolute, out_off from the window's first byte
  size_t used = 0;                                // bytes of whole blocks
  uint64_t total = 0;                             // inflated bytes
  ~DevInflated() {
    for (void* p : {(void*)in, (void*)out, (void*)blocks, (void*)status, (void*)bitmap}) if (p) cudaFree(p);
  }
};

// BGZF framing of `bgzf` (file bytes from `file_off`) and the compressed bytes' device buffer
int inflate_frame(ngsq_engine* e, const uint8_t* bgzf, size_t nbytes, uint64_t file_off, DevInflated& D) {
  uint32_t n = 0;
  int rc = ngsq_bgzf_walk(bgzf, nbytes, file_off, nullptr, 0, &n, &D.used);
  if (rc) return fail(e, rc, "malformed BGZF framing");
  std::vector<ngsq_block> blk(n);
  ngsq_bgzf_walk(bgzf, nbytes, file_off, blk.data(), n, &n, &D.used);
  CU(cudaMalloc(&D.in, D.used + 512));
  for (auto& b : blk) {
    if (b.csize < b.hdr_len + 8 || b.isize > 65536) return fail(e, NGSQ_E_BAD_BLOCK, "malformed BGZF block");
    if (!b.isize) continue;
    D.hb.push_back({(uint64_t)(uintptr_t)D.in + (b.coffset - file_off) + b.hdr_len, D.total, b.csize - b.hdr_len - 8, b.isize, b.coffset});
    D.total += b.isize;
  }
  return NGSQ_OK;
}

// K2 over the framed blocks; fails with the first block that does not inflate
int inflate_run(ngsq_engine* e, const uint8_t* bgzf, DevInflated& D) {
  if (D.hb.empty()) return NGSQ_OK;
  cudaStream_t s = e->s_copy;
  const size_t nb = D.hb.size();
  CU(cudaMalloc(&D.out, D.total + 64));
  CU(cudaMalloc(&D.blocks, nb * sizeof(BlockDesc)));
  CU(cudaMalloc(&D.status, nb * 4 + 64));
  CU(cudaMalloc(&D.bitmap, nb * kBitmapWords * 4));
  CU(cudaMemcpyAsync(D.in, bgzf, D.used, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(D.blocks, D.hb.data(), nb * sizeof(BlockDesc), cudaMemcpyHostToDevice, s));
  int rc = launch_inflate(e, D.blocks, (uint32_t)nb, D.out, D.status + nb, D.status, D.bitmap, s);
  if (rc) return rc;
  std::vector<uint32_t> st(nb);
  CU(cudaMemcpyAsync(st.data(), D.status, nb * 4, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  for (size_t i = 0; i < nb; ++i)
    if (st[i]) return fail(e, NGSQ_E_BAD_BLOCK, "block %zu failed to inflate (status %u)", i, st[i]);
  return NGSQ_OK;
}

}  // namespace

extern "C" {

namespace {
// Host copies of the group buffer after ngsq_finish / ngsq_reduce: the counters and lengths, then each group's quality rows
int fetch_groups(ngsq_engine* e, cudaStream_t s) {
  const uint64_t ng = (uint64_t)e->rg_n + 1, head = ng * (kGroupSums + 1);
  e->h_grp_sums.assign(ng * kGroupSums, 0);
  e->h_grp_qlen.assign(ng, 0);
  CU(cudaMemcpyAsync(e->h_grp_sums.data(), e->d_grp, ng * kGroupSums * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(e->h_grp_qlen.data(), e->d_grp + ng * kGroupSums, ng * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  e->h_grp_qual.assign(ng, {});
  for (uint64_t g = 0; g < ng; ++g) {
    e->h_grp_qlen[g] = std::min<uint64_t>(e->h_grp_qlen[g], e->grp_rows);
    e->h_grp_qual[g].resize(e->h_grp_qlen[g] * 94);
    if (e->h_grp_qlen[g])
      CU(cudaMemcpyAsync(e->h_grp_qual[g].data(), e->d_grp + head + g * e->grp_rows * 94, e->h_grp_qlen[g] * 94 * 8, cudaMemcpyDeviceToHost, s));
  }
  CU(cudaStreamSynchronize(s));
  return NGSQ_OK;
}
}  // namespace

int ngsq_version(void) { return NGSQ_VERSION; }

const char* ngsq_last_error(ngsq_engine* e) { return e ? e->err.c_str() : g_create_err.c_str(); }

int ngsq_create(int device, const ngsq_config* cfg, ngsq_engine** out) {
  ngsq_engine* e = nullptr;
  if (!out) return fail(e, NGSQ_E_ARG, "out is NULL");
  *out = nullptr;
  int n_dev = 0;
  cudaError_t rc = cudaGetDeviceCount(&n_dev);
  if (rc != cudaSuccess || n_dev == 0)
    return fail(e, NGSQ_E_CUDA, "no CUDA device available (%s); the ngs-cuda engine has no CPU fallback", cudaGetErrorString(rc));
  if (device < 0 || device >= n_dev) return fail(e, NGSQ_E_ARG, "device %d out of range (%d devices)", device, n_dev);
  if (cfg && (cfg->flags & NGSQ_F_INDEX) && (cfg->flags & NGSQ_F_INDEX_PART))
    return fail(e, NGSQ_E_ARG, "NGSQ_F_INDEX_PART is set instead of NGSQ_F_INDEX, not with it");
  if (cfg && (cfg->flags & NGSQ_F_INDEX_CSI) && !(cfg->flags & (NGSQ_F_INDEX | NGSQ_F_INDEX_PART)))
    return fail(e, NGSQ_E_ARG, "NGSQ_F_INDEX_CSI selects the format of NGSQ_F_INDEX or NGSQ_F_INDEX_PART: set one of them with it");
  if (cfg && (cfg->flags & (NGSQ_F_INDEX | NGSQ_F_INDEX_PART)) && cfg->max_records)
    return fail(e, NGSQ_E_ARG, "NGSQ_F_INDEX cannot be combined with max_records: an index covers every record of the file");
  if (cfg && (cfg->flags & NGSQ_F_READ_GROUPS) && !(cfg->flags & NGSQ_F_RECORD_FACETS))
    return fail(e, NGSQ_E_ARG, "NGSQ_F_READ_GROUPS splits the record facets by read group: set NGSQ_F_RECORD_FACETS with it");
  ngsq_engine* ne = new ngsq_engine();
  ne->device = device;
  if (cfg) memcpy(&ne->cfg, cfg, std::min<size_t>(cfg->struct_size ? cfg->struct_size : sizeof(ngsq_config), sizeof(ngsq_config)));
  if (!ne->cfg.flags) ne->cfg.flags = NGSQ_F_RECORD_FACETS | NGSQ_F_COVERAGE;
  if (const char* v = getenv("NGSQ_TRACE")) ne->trace = atoi(v) != 0;
  ne->headroom = ne->cfg.carry_bytes ? ((ne->cfg.carry_bytes + 63u) & ~63u) : kDefaultHeadroom;
  e = ne;
  auto bail = [&](int code) { std::string m = e->err; ngsq_destroy(e); g_create_err = m; return code; };
#define CUC(call) do { cudaError_t _r = (call); if (_r != cudaSuccess) { fail(e, NGSQ_E_CUDA, "%s: %s", #call, cudaGetErrorString(_r)); return bail(NGSQ_E_CUDA); } } while (0)
  CUC(cudaSetDevice(device));
  cudaDeviceProp prop;
  CUC(cudaGetDeviceProperties(&prop, device));
  e->n_sm = prop.multiProcessorCount;
  CUC(cudaStreamCreateWithFlags(&e->s_copy, cudaStreamNonBlocking));
  {
    // Which kernel gets an SM when several wait for one: the scan stream's first (short kernels that gate the reuse of a
    // slot), inflate next, the CRC check last (numerically lower = higher priority)
    int prio_low = 0, prio_high = 0;
    CUC(cudaDeviceGetStreamPriorityRange(&prio_low, &prio_high));
    const int prio_mid = prio_high < prio_low - 1 ? prio_low - 1 : prio_high;
    CUC(cudaStreamCreateWithPriority(&e->s_scan, cudaStreamNonBlocking, prio_high));
    CUC(cudaStreamCreateWithPriority(&e->s_comp, cudaStreamNonBlocking, prio_mid));
    CUC(cudaStreamCreateWithPriority(&e->s_aux, cudaStreamNonBlocking, prio_low));
  }
  for (cudaEvent_t* ev : {&e->ev_start, &e->ev_a, &e->ev_b, &e->ev_d, &e->ev_e, &e->ev_f, &e->ev_g}) CUC(cudaEventCreate(ev));
  CUC(cudaMalloc(&e->d_queue, 64));
  CUC(cudaMalloc(&e->d_state, sizeof(RunState)));
  CUC(cudaHostAlloc((void**)&e->h_state, sizeof(RunState), cudaHostAllocDefault));
  CUC(cudaHostAlloc((void**)&e->h_prog, kProgSlots * 16, cudaHostAllocDefault));
  if (ix_on(e)) {
    CUC(cudaMalloc(&e->d_ix, sizeof(IndexState)));
    CUC(cudaMalloc(&e->d_ix_ovf, kIndexOverflowCap * (ix_csi(e) ? sizeof(IndexOvf) : sizeof(IndexRun))));
    CUC(cudaHostAlloc((void**)&e->h_ix_probe, 16, cudaHostAllocDefault));
  }
  CUC(cudaMalloc(&e->d_crc_tables, sizeof(CrcTables)));
  // opt-in shared memory sizes are per device: set them for this engine's device (several engines of
  // one process may sit on different GPUs)
  CUC(cudaFuncSetAttribute(crc32_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kCrcSmem));
  CUC(cudaFuncSetAttribute(inflate_decode_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDecSmem));
  e->facet_smem = (size_t)qual_table_bytes(kQualSmemPositions) * (kFacetThreads / 32) + (size_t)(kTlenPad + kGcPad + kCigWords) * 4;
  CUC(cudaFuncSetAttribute(facets_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->facet_smem));
  CUC(cudaFuncSetAttribute(qual_tiles_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTileSmem));
  CUC(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&e->facet_occ, facets_kernel, kFacetThreads, e->facet_smem));
  if (e->facet_occ < 1) e->facet_occ = 1;
  if (rg_on(e)) {
    e->rg_smem = rg_facets_smem(kFacetThreads / 32);
    CUC(cudaFuncSetAttribute(rg_facets_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)e->rg_smem));
    CUC(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&e->rg_occ, rg_facets_kernel, kFacetThreads, e->rg_smem));
    if (e->rg_occ < 1) e->rg_occ = 1;
    CUC(cudaMalloc(&e->d_rg_total, 4));
  }
  {
    CrcTables t;
    crc_make_tables(t);
    CUC(cudaMemcpy(e->d_crc_tables, &t, sizeof t, cudaMemcpyHostToDevice));
  }
  if (e->cfg.reserve_compressed) {
    // the caller keeps the whole compressed shard on the device (one segment, no recycling needed)
    uint8_t* p = nullptr;
    size_t cap = e->cfg.reserve_compressed + (e->cfg.reserve_compressed >> 6) + 4096;  // room for 16-byte chunk padding
    CUC(cudaMalloc(&p, cap + 512));
    e->comp_segs.push_back({p, cap, 0, 0});
    e->comp_total = cap;
  }
#undef CUC
  *out = e;
  return NGSQ_OK;
}

void ngsq_destroy(ngsq_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  cudaDeviceSynchronize();
  if (e->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(e->comm);
  for (auto& c : e->chunks) cudaEventDestroy(c.copied);
  for (auto& p : e->waves) for (cudaEvent_t x : {p.begin, p.decoded_from, p.decoded, p.resolved, p.scan_begin, p.begun, p.scan_end, p.facets_end, p.crc_begin, p.crc_end}) cudaEventDestroy(x);
  for (cudaEvent_t ev : {e->ev_start, e->ev_a, e->ev_b, e->ev_d, e->ev_e, e->ev_f, e->ev_g}) if (ev) cudaEventDestroy(ev);
  void* ptrs[] = {e->d_ref_len, e->d_cov_enabled, e->d_diff_base, e->d_cov_slot, e->d_diff, e->d_tile, e->d_tile_off, e->d_tile_sum, e->d_res, e->d_long, e->d_slot[0], e->d_slot[1],
                  e->d_blocks_all, e->d_crc_all, e->d_wstatus[0], e->d_wstatus[1], e->d_first, e->d_landed, e->d_count, e->d_base,
                  e->d_bitmap, e->d_rec, e->d_mark, e->d_queue, e->d_state, e->d_crc_tables};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (e->h_state) cudaFreeHost(e->h_state);
  if (e->h_prog) cudaFreeHost(e->h_prog);
  for (auto& ps : e->pin_slabs) cudaFreeHost(ps.p);
  for (void* p : e->ed_allocs) cudaFree(p);
  for (void* p : {(void*)e->d_ed_contigs, (void*)e->d_ed_refs, (void*)e->d_ed_alts, (void*)e->d_ed_res}) if (p) cudaFree(p);
  for (void* p : e->ft_allocs) cudaFree(p);
  for (void* p : {(void*)e->d_ft_contigs, (void*)e->d_ft_res}) if (p) cudaFree(p);
  for (void* p : {(void*)e->d_rg_ids, (void*)e->d_rg_id_off, (void*)e->d_rg_table, (void*)e->d_grp, (void*)e->d_rg_of, (void*)e->d_rg_order,
                  (void*)e->d_rg_count, (void*)e->d_rg_cursor, (void*)e->d_rg_total}) if (p) cudaFree(p);
  for (auto& w : e->ix_waves) cudaEventDestroy(w.done);
  for (void* p : {(void*)e->d_ix, (void*)e->d_ix_runs[0], (void*)e->d_ix_runs[1], (void*)e->d_ix_ovf, (void*)e->d_ix_win_base, (void*)e->d_ix_win_n,
                  (void*)e->d_ix_win, (void*)e->d_ix_maxw, (void*)e->d_ix_counts}) if (p) cudaFree(p);
  if (e->h_ix_probe) cudaFreeHost(e->h_ix_probe);
  for (auto& sg : e->comp_segs) cudaFree(sg.ptr);
  if (e->s_copy) cudaStreamDestroy(e->s_copy);
  if (e->s_comp) cudaStreamDestroy(e->s_comp);
  if (e->s_aux) cudaStreamDestroy(e->s_aux);
  if (e->s_scan) cudaStreamDestroy(e->s_scan);
  delete e;
}

int ngsq_reset(ngsq_engine* e) {
  if (!e) return NGSQ_E_ARG;
  CU(cudaSetDevice(e->device));
  CU(cudaStreamSynchronize(e->s_copy));
  CU(cudaStreamSynchronize(e->s_comp));
  CU(cudaStreamSynchronize(e->s_scan));
  CU(cudaStreamSynchronize(e->s_aux));
  for (auto& c : e->chunks) cudaEventDestroy(c.copied);
  e->chunks.clear();
  e->launched = 0;
  for (auto& p : e->waves) for (cudaEvent_t x : {p.begin, p.decoded_from, p.decoded, p.resolved, p.scan_begin, p.begun, p.scan_end, p.facets_end, p.crc_begin, p.crc_end}) cudaEventDestroy(x);
  e->waves.clear();
  e->h_blocks.clear(); e->h_crc.clear();
  for (auto& sg : e->comp_segs) { sg.used = 0; sg.blocks_end = 0; }
  for (auto& ps : e->pin_slabs) ps.used = 0;
  e->out_used = 0; e->comp_bytes_total = 0; e->other_launches = 0;
  e->start_resolved = e->end_resolved = false;
  e->file_b0 = 0; e->awaiting_range = false;
  e->prog_seen = 0; e->prog_records = 0;
  e->host_ms.clear();
  // rows of the quality table the next run has to clear; a run that never reached ngsq_finish may have touched any
  e->qpos_dirty = (e->run_started && !e->finished) ? e->qpos_cap : std::max(e->qpos_dirty, e->h_qpos);
  e->run_started = false; e->finished = false;
  e->h_res.clear(); e->h_qpos = 0;
  e->h_ed_res.clear();
  e->h_ft_res.clear();
  e->h_grp_sums.clear(); e->h_grp_qlen.clear(); e->h_grp_qual.clear();
  e->rg_sel = -1;  // the IDs, the table and the group buffer are kept
  for (auto& w : e->ix_waves) cudaEventDestroy(w.done);
  e->ix_waves.clear();
  e->ix_drained.clear();  // pinned memory of the pin slabs, released above
  e->data_end_coff = 0;
  e->ix_bytes.clear();
  e->ix = IxHost{};
  e->ix_part_ok = false;
  e->split_merged = false;  // the split set itself is kept
  memset(&e->stats, 0, sizeof e->stats);
  return NGSQ_OK;
}

int ngsq_set_references(ngsq_engine* e, uint32_t n_ref, const uint32_t* ref_len, const uint8_t* coverage_enabled) {
  if (!e || (n_ref && (!ref_len || !coverage_enabled))) return fail(e, NGSQ_E_ARG, "bad references");
  if (e->run_started) return fail(e, NGSQ_E_ARG, "ngsq_set_references must precede the first submit");
  if (ix_on(e) && ix_csi(e)) {
    uint32_t max_len = 0;
    for (uint32_t c = 0; c < n_ref; ++c) max_len = std::max(max_len, ref_len[c]);
    const uint32_t depth = e->ix_depth_req ? e->ix_depth_req : ix_csi_default_depth(max_len, e->ix_min_shift);
    for (uint32_t c = 0; c < n_ref; ++c)
      if (ref_len[c] > ix_csi_max_end(e->ix_min_shift, depth))
        return fail(e, NGSQ_E_ARG, "reference %u is %u bases long: a CSI of min_shift %u and depth %u addresses at most 2^%u bases", c,
                    ref_len[c], e->ix_min_shift, depth, e->ix_min_shift + 3 * depth);
    e->ix_depth = depth;
  } else if (ix_on(e))
    for (uint32_t c = 0; c < n_ref; ++c)
      if (ref_len[c] >= kIxMaxEnd)
        return fail(e, NGSQ_E_ARG, "reference %u is %u bases long: a BAI addresses fewer than 2^29 bases (index this file as CSI)", c, ref_len[c]);
  CU(cudaSetDevice(e->device));
  e->n_ref = n_ref;
  e->ref_len.assign(ref_len, ref_len + n_ref);
  e->cov_enabled.assign(coverage_enabled, coverage_enabled + n_ref);
  if (!(e->cfg.flags & NGSQ_F_COVERAGE)) std::fill(e->cov_enabled.begin(), e->cov_enabled.end(), 0);
  e->diff_base.assign(n_ref, 0);
  e->tile_off.assign(n_ref, 0);
  e->split_ref.assign(n_ref, 0);
  e->n_split = 0;
  e->split_merged = false;
  e->layout_agreed = false;
  uint64_t elems = 0, tiles = 0;
  uint32_t max_tiles = 1;
  for (uint32_t c = 0; c < n_ref; ++c) {
    e->diff_base[c] = elems;
    e->tile_off[c] = (uint32_t)tiles;
    if (e->cov_enabled[c]) {
      elems += ((uint64_t)ref_len[c] + 2 + 3) & ~3ull;  // keep every contig 16-byte aligned
      const uint32_t nt = (uint32_t)(((uint64_t)ref_len[c] + 1 + kCovTile - 1) / kCovTile);
      max_tiles = std::max<uint32_t>(max_tiles, nt);
      tiles += nt;
    }
  }
  e->tile_total = tiles ? tiles : 1;
  for (void* p : {(void*)e->d_ref_len, (void*)e->d_cov_enabled, (void*)e->d_diff_base, (void*)e->d_cov_slot, (void*)e->d_diff, (void*)e->d_tile, (void*)e->d_tile_off, (void*)e->d_tile_sum}) if (p) cudaFree(p);
  e->d_ref_len = nullptr; e->d_cov_enabled = nullptr; e->d_diff_base = nullptr; e->d_cov_slot = nullptr; e->d_diff = nullptr; e->d_tile = nullptr;
  e->d_tile_off = nullptr; e->d_tile_sum = nullptr;
  size_t nr = n_ref ? n_ref : 1;
  CU(cudaMalloc(&e->d_ref_len, nr * 4));
  CU(cudaMalloc(&e->d_cov_enabled, nr));
  CU(cudaMalloc(&e->d_diff_base, nr * 8));
  CU(cudaMalloc(&e->d_cov_slot, nr * 4));
  CU(cudaMalloc(&e->d_tile_off, nr * 4));
  CU(cudaMalloc(&e->d_tile_sum, e->tile_total * 4));
  if (n_ref) {
    CU(cudaMemcpy(e->d_tile_off, e->tile_off.data(), n_ref * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->d_ref_len, e->ref_len.data(), n_ref * 4, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->d_cov_enabled, e->cov_enabled.data(), n_ref, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(e->d_diff_base, e->diff_base.data(), n_ref * 8, cudaMemcpyHostToDevice));
  }
  e->diff_elems = elems;
  if (elems) {
    cudaError_t rc = cudaMalloc(&e->d_diff, elems * 4 + 64);
    if (rc != cudaSuccess) return fail(e, NGSQ_E_NOMEM, "cudaMalloc difference arrays (%llu bytes): %s", (unsigned long long)elems * 4, cudaGetErrorString(rc));
  }
  CU(cudaMalloc(&e->d_tile, (size_t)max_tiles * 8));
  e->tile_cap = max_tiles;
  // a new header means a new layout: the buffer is rebuilt (and zeroed) with the configured quality capacity
  const uint32_t qcap = std::max(e->qpos_cap, e->cfg.quality_positions ? e->cfg.quality_positions : kDefaultQualPositions);
  e->qpos_cap = 0;
  e->res_words = 0;
  e->res_cap_words = 0;
  if (e->d_res) { cudaFree(e->d_res); e->d_res = nullptr; }
  e->qpos_dirty = 0;
  int rc = ensure_res(e, qcap, false);
  if (rc) return rc;
  if (e->cfg.flags & NGSQ_F_EDITS) {
    // sequences loaded for an earlier header are dropped; per-position counters cover 0..=L of every contig
    for (void* p : e->ed_allocs) cudaFree(p);
    e->ed_allocs.clear();
    for (void* p : {(void*)e->d_ed_contigs, (void*)e->d_ed_refs, (void*)e->d_ed_alts}) if (p) cudaFree(p);
    e->d_ed_contigs = nullptr; e->d_ed_refs = nullptr; e->d_ed_alts = nullptr;
    e->ed_contigs.assign(n_ref, EditsContig{});
    uint64_t total = 0;
    for (uint32_t c = 0; c < n_ref; ++c) {
      e->ed_contigs[c].hdr_len = ref_len[c];
      e->ed_contigs[c].pos_off = total;
      total += (uint64_t)ref_len[c] + 1;
    }
    e->ed_pos_total = total;
    CU(cudaMalloc(&e->d_ed_contigs, nr * sizeof(EditsContig)));
    if (n_ref) CU(cudaMemcpy(e->d_ed_contigs, e->ed_contigs.data(), n_ref * sizeof(EditsContig), cudaMemcpyHostToDevice));
    if (total) {
      cudaError_t r1 = cudaMalloc(&e->d_ed_refs, total * 4), r2 = r1 == cudaSuccess ? cudaMalloc(&e->d_ed_alts, total * 4) : r1;
      if (r2 != cudaSuccess) return fail(e, NGSQ_E_NOMEM, "cudaMalloc per-position edit counters (%llu bytes): %s", (unsigned long long)total * 8, cudaGetErrorString(r2));
    }
    if (!e->d_ed_res) CU(cudaMalloc(&e->d_ed_res, E_WORDS * 8));
  }
  if (e->cfg.flags & NGSQ_F_FEATURES) {
    for (void* p : e->ft_allocs) cudaFree(p);
    e->ft_allocs.clear();
    if (e->d_ft_contigs) cudaFree(e->d_ft_contigs);
    e->d_ft_contigs = nullptr;
    e->ft_contigs.assign(n_ref, FeatureContig{});
    e->ft_model_set = false;
    CU(cudaMalloc(&e->d_ft_contigs, nr * sizeof(FeatureContig)));
    if (n_ref) CU(cudaMemcpy(e->d_ft_contigs, e->ft_contigs.data(), n_ref * sizeof(FeatureContig), cudaMemcpyHostToDevice));
    if (!e->d_ft_res) CU(cudaMalloc(&e->d_ft_res, F_WORDS * 8));
  }
  if (ix_on(e)) {
    // window table per reference: windows 0 ..= L >> 14 (BAI) or L >> min_shift (CSI); reads overhanging the end go to the
    // overflow list
    e->ix_win_base.assign(n_ref, 0);
    e->ix_win_n.assign(n_ref, 0);
    uint64_t total = 0;
    for (uint32_t c = 0; c < n_ref; ++c) {
      e->ix_win_base[c] = total;
      e->ix_win_n[c] = (ref_len[c] >> (ix_csi(e) ? e->ix_min_shift : kIxWindowShift)) + 1;
      total += e->ix_win_n[c];
    }
    e->ix_win_total = total;
    for (void* p : {(void*)e->d_ix_win_base, (void*)e->d_ix_win_n, (void*)e->d_ix_win, (void*)e->d_ix_maxw, (void*)e->d_ix_counts}) if (p) cudaFree(p);
    CU(cudaMalloc(&e->d_ix_win_base, nr * 8));
    CU(cudaMalloc(&e->d_ix_win_n, nr * 4));
    CU(cudaMalloc(&e->d_ix_win, std::max<uint64_t>(total, 1) * 8));
    CU(cudaMalloc(&e->d_ix_maxw, nr * 4));
    CU(cudaMalloc(&e->d_ix_counts, nr * 16));
    if (n_ref) {
      CU(cudaMemcpy(e->d_ix_win_base, e->ix_win_base.data(), n_ref * 8, cudaMemcpyHostToDevice));
      CU(cudaMemcpy(e->d_ix_win_n, e->ix_win_n.data(), n_ref * 4, cudaMemcpyHostToDevice));
    }
  }
  return NGSQ_OK;
}

int ngsq_set_feature_model(ngsq_engine* e, const uint8_t slot_class[5], const uint8_t* primary) {
  if (!e || !slot_class || (e->n_ref && !primary)) return fail(e, NGSQ_E_ARG, "bad feature model");
  if (!(e->cfg.flags & NGSQ_F_FEATURES)) return fail(e, NGSQ_E_ARG, "the engine was created without NGSQ_F_FEATURES");
  if (e->ft_contigs.size() != e->n_ref) return fail(e, NGSQ_E_ARG, "ngsq_set_feature_model must follow ngsq_set_references");
  if (e->run_started) return fail(e, NGSQ_E_ARG, "ngsq_set_feature_model must precede the first submit");
  for (int j = 0; j < 5; ++j)
    if (slot_class[j] > j || slot_class[slot_class[j]] != slot_class[j]) return fail(e, NGSQ_E_ARG, "slot_class[%d] must name the first slot with the same feature name", j);
  CU(cudaSetDevice(e->device));
  memcpy(e->ft_slot_class, slot_class, 5);
  for (uint32_t c = 0; c < e->n_ref; ++c) e->ft_contigs[c].primary = primary[c] ? 1u : 0u;
  if (e->n_ref) CU(cudaMemcpy(e->d_ft_contigs, e->ft_contigs.data(), e->n_ref * sizeof(FeatureContig), cudaMemcpyHostToDevice));
  e->ft_model_set = true;
  return NGSQ_OK;
}

int ngsq_set_features(ngsq_engine* e, uint32_t ref, uint32_t n, const uint32_t* start, const uint32_t* stop, const uint8_t* cls) {
  if (!e || (n && (!start || !stop || !cls))) return fail(e, NGSQ_E_ARG, "bad features");
  if (!(e->cfg.flags & NGSQ_F_FEATURES)) return fail(e, NGSQ_E_ARG, "the engine was created without NGSQ_F_FEATURES");
  if (ref >= e->n_ref || e->ft_contigs.size() != e->n_ref) return fail(e, NGSQ_E_ARG, "ngsq_set_features: reference %u is not in the header given to ngsq_set_references", ref);
  if (e->run_started) return fail(e, NGSQ_E_ARG, "ngsq_set_features must precede the first submit");
  CU(cudaSetDevice(e->device));
  FeatureContig& C = e->ft_contigs[ref];
  for (int k = 0; k < 5; ++k) if (C.n[k]) return fail(e, NGSQ_E_ARG, "reference %u already has features", ref);
  std::vector<uint32_t> a[5], b[5];
  for (uint32_t i = 0; i < n; ++i) {
    if (cls[i] > 4) return fail(e, NGSQ_E_ARG, "feature class %u out of range", cls[i]);
    if (start[i] > stop[i]) return fail(e, NGSQ_E_ARG, "feature %u has start > end (%u > %u): not supported by the counting lookup", i, start[i], stop[i]);
    a[cls[i]].push_back(start[i]);
    b[cls[i]].push_back(stop[i]);
  }
  for (int k = 0; k < 5; ++k) {
    if (a[k].empty()) continue;
    std::sort(a[k].begin(), a[k].end());
    std::sort(b[k].begin(), b[k].end());
    uint32_t *da = nullptr, *db = nullptr;
    const size_t bytes = a[k].size() * 4;
    cudaError_t rc = cudaMalloc(&da, bytes);
    if (rc == cudaSuccess) { e->ft_allocs.push_back(da); rc = cudaMalloc(&db, bytes); }
    if (rc != cudaSuccess) return fail(e, NGSQ_E_NOMEM, "cudaMalloc features (%zu bytes): %s", bytes, cudaGetErrorString(rc));
    e->ft_allocs.push_back(db);
    CU(cudaMemcpy(da, a[k].data(), bytes, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(db, b[k].data(), bytes, cudaMemcpyHostToDevice));
    C.starts[k] = da; C.stops[k] = db; C.n[k] = (uint32_t)a[k].size();
  }
  CU(cudaMemcpy(e->d_ft_contigs + ref, &C, sizeof C, cudaMemcpyHostToDevice));
  return NGSQ_OK;
}

int ngsq_set_reference_bases(ngsq_engine* e, uint32_t ref, const uint8_t* letters, uint64_t n) {
  if (!e || (!letters && n)) return fail(e, NGSQ_E_ARG, "bad reference bases");
  if (!(e->cfg.flags & NGSQ_F_EDITS)) return fail(e, NGSQ_E_ARG, "the engine was created without NGSQ_F_EDITS");
  if (ref >= e->n_ref || e->ed_contigs.size() != e->n_ref) return fail(e, NGSQ_E_ARG, "ngsq_set_reference_bases: reference %u is not in the header given to ngsq_set_references", ref);
  if (e->run_started) return fail(e, NGSQ_E_ARG, "ngsq_set_reference_bases must precede the first submit");
  if (e->ed_contigs[ref].codes) return fail(e, NGSQ_E_ARG, "reference %u already has a sequence", ref);
  CU(cudaSetDevice(e->device));
  const uint64_t words = n / 32 + 1;
  std::vector<uint8_t> codes(n + 1);
  std::vector<uint32_t> bits(words), prefix(words);
  edits_encode(letters, n, codes.data(), bits.data(), prefix.data());
  uint8_t* d_codes = nullptr;
  uint32_t *d_bits = nullptr, *d_prefix = nullptr;
  cudaError_t rc = cudaMalloc(&d_codes, n + 64);
  if (rc == cudaSuccess) { e->ed_allocs.push_back(d_codes); rc = cudaMalloc(&d_bits, words * 4); }
  if (rc == cudaSuccess) { e->ed_allocs.push_back(d_bits); rc = cudaMalloc(&d_prefix, words * 4); }
  if (rc != cudaSuccess) return fail(e, NGSQ_E_NOMEM, "cudaMalloc reference sequence (%llu bases): %s", (unsigned long long)n, cudaGetErrorString(rc));
  e->ed_allocs.push_back(d_prefix);
  CU(cudaMemcpy(d_codes, codes.data(), n, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(d_bits, bits.data(), words * 4, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(d_prefix, prefix.data(), words * 4, cudaMemcpyHostToDevice));
  EditsContig& C = e->ed_contigs[ref];
  C.codes = d_codes; C.bad_bits = d_bits; C.bad_prefix = d_prefix; C.code_len = n;
  CU(cudaMemcpy(e->d_ed_contigs + ref, &C, sizeof C, cudaMemcpyHostToDevice));
  return NGSQ_OK;
}

int ngsq_set_range(ngsq_engine* e, uint64_t first_rec_voffset, uint64_t end_voffset) {
  if (!e) return NGSQ_E_ARG;
  if (e->launched && !e->awaiting_range) return fail(e, NGSQ_E_ARG, "ngsq_set_range must precede the first submit of a run");
  if ((e->cfg.flags & NGSQ_F_INDEX) && end_voffset)
    return fail(e, NGSQ_E_ARG, "NGSQ_F_INDEX needs end_voffset 0: an index covers the whole file from its first record");
  if (e->awaiting_range) {  // the next file of the run: its blocks start behind the last one's
    e->file_b0 = (uint32_t)e->h_blocks.size();
    e->awaiting_range = false;
  }
  e->first_voff = first_rec_voffset;
  e->end_voff = end_voffset;
  e->range_set = true;
  e->start_resolved = e->end_resolved = false;
  return NGSQ_OK;
}

int ngsq_bgzf_walk(const uint8_t* p, size_t n, uint64_t file_off, ngsq_block* out, uint32_t cap, uint32_t* n_blocks, size_t* consumed) {
  size_t o = 0;
  uint32_t k = 0;
  while (n - o >= 18) {
    const uint8_t* h = p + o;
    if (h[0] != 0x1f || h[1] != 0x8b || h[2] != 8 || !(h[3] & 4)) return NGSQ_E_BAD_BLOCK;
    uint32_t xlen = h[10] | (h[11] << 8);
    if (n - o < 12 + xlen) break;
    uint32_t bsize = 0;
    bool found = false;
    for (uint32_t q = 0; q + 4 <= xlen;) {
      const uint8_t* s = h + 12 + q;
      uint32_t slen = s[2] | (s[3] << 8);
      if (s[0] == 'B' && s[1] == 'C' && slen == 2 && q + 6 <= xlen) { bsize = s[4] | (s[5] << 8); found = true; }
      q += 4 + slen;
    }
    if (!found) return NGSQ_E_BAD_BLOCK;
    size_t total = (size_t)bsize + 1;
    if (total < 12 + xlen + 8) return NGSQ_E_BAD_BLOCK;
    if (n - o < total) break;
    if (out) {
      if (k >= cap) break;
      ngsq_block& b = out[k];
      b.coffset = file_off + o;
      b.hdr_len = 12 + xlen;
      b.csize = (uint32_t)total;
      memcpy(&b.crc32, h + total - 8, 4);
      memcpy(&b.isize, h + total - 4, 4);
    }
    ++k;
    o += total;
  }
  if (n_blocks) *n_blocks = k;
  if (consumed) *consumed = o;
  return NGSQ_OK;
}

int ngsq_submit(ngsq_engine* e, const uint8_t* bgzf, size_t nbytes, uint64_t file_off) {
  if (!e || !bgzf) return fail(e, NGSQ_E_ARG, "bad submit arguments");
  if (e->finished) return fail(e, NGSQ_E_ARG, "submit after finish; call ngsq_reset");
  if (!e->range_set) return fail(e, NGSQ_E_ARG, "ngsq_set_range must precede the first submit");
  if (e->awaiting_range) return fail(e, NGSQ_E_ARG, "ngsq_set_range must follow ngsq_next_file before the next file's first submit");
  CU(cudaSetDevice(e->device));
  uint32_t n = 0;
  size_t used = 0;
  int rc = ngsq_bgzf_walk(bgzf, nbytes, file_off, nullptr, 0, &n, &used);
  if (rc) return fail(e, rc, "malformed BGZF framing in chunk at file offset %llu", (unsigned long long)file_off);
  if (used != nbytes) return fail(e, NGSQ_E_TRUNCATED, "chunk at file offset %llu ends inside a BGZF block (%zu of %zu bytes are whole blocks)", (unsigned long long)file_off, used, nbytes);
  std::vector<ngsq_block> blk(n);
  ngsq_bgzf_walk(bgzf, nbytes, file_off, blk.data(), n, &n, &used);
  rc = start_run(e);
  if (rc) return rc;
  uint8_t* dst = nullptr;
  rc = acquire_comp(e, nbytes, &dst);
  if (rc) return rc;
  CU(cudaMemcpyAsync(dst, bgzf, nbytes, cudaMemcpyHostToDevice, e->s_copy));
  e->comp_bytes_total += nbytes;
  const uint32_t first_new = (uint32_t)e->h_blocks.size();
  rc = append_blocks(e, blk.data(), n, (uint64_t)(uintptr_t)dst, file_off);
  if (rc) return rc;
  rc = upload_descriptors(e, first_new, (uint32_t)e->h_blocks.size());
  if (rc) return rc;
  cudaEvent_t ev;
  CU(cudaEventCreateWithFlags(&ev, e->trace ? cudaEventDefault : cudaEventDisableTiming));
  CU(cudaEventRecord(ev, e->s_copy));
  e->chunks.push_back({ev, (uint32_t)e->h_blocks.size()});
  e->comp_segs.back().blocks_end = (uint32_t)e->h_blocks.size();
  // inflate in whole waves; the copy of the next chunk overlaps the kernels of this one
  const uint32_t quantum = launch_quantum(e), total = (uint32_t)e->h_blocks.size(), pending = total - e->launched;
  // Every wave costs one decode round (~18 ms on a B200 whatever its size), and at 55 GB/s of PCIe the GPU work of a
  // shard takes as long as its copy: fewer, full waves win.  A smaller first wave (earlier start) and a cut-off last wave
  // (shorter tail) were measured and each cost a round more than it saved (profiles/round2_e2e_timeline.md); callers
  // whose copies are the slower side can still ask for a short tail with ngsq_flush.
  if (pending >= quantum) return launch_pending(e, e->launched + pending / quantum * quantum, false);
  return NGSQ_OK;
}

int ngsq_flush(ngsq_engine* e) {
  if (!e) return NGSQ_E_ARG;
  if (e->finished) return NGSQ_OK;
  CU(cudaSetDevice(e->device));
  return launch_pending(e, (uint32_t)e->h_blocks.size(), false);
}

int ngsq_next_file(ngsq_engine* e) {
  if (!e) return NGSQ_E_ARG;
  if (e->finished) return fail(e, NGSQ_E_ARG, "ngsq_next_file after finish; call ngsq_reset");
  if (ix_on(e)) return fail(e, NGSQ_E_ARG, "ngsq_next_file: an index (NGSQ_F_INDEX, NGSQ_F_INDEX_PART) describes one file");
  if (e->cfg.max_records) return fail(e, NGSQ_E_ARG, "ngsq_next_file: max_records counts the records of one file in its order");
  if (!e->range_set || e->awaiting_range) return fail(e, NGSQ_E_ARG, "ngsq_next_file: call ngsq_set_range for the file first");
  CU(cudaSetDevice(e->device));
  int rc = start_run(e);
  if (rc) return rc;
  // the file's last wave: a record that runs past its end is a truncation, and no later wave holds blocks of this file
  const uint32_t nb = (uint32_t)e->h_blocks.size();
  if ((rc = launch_pending(e, nb, true))) return rc;
  if (nb > e->file_b0) {
    if (!e->start_resolved && (e->first_voff & 0xFFFF)) return fail(e, NGSQ_E_ARG, "virtual offset %llu is beyond the submitted data", (unsigned long long)e->first_voff);
    if (e->end_voff && !e->end_resolved && (e->end_voff & 0xFFFF)) return fail(e, NGSQ_E_ARG, "virtual offset %llu is beyond the submitted data", (unsigned long long)e->end_voff);
  }
  if (!e->waves.empty()) {
    // behind the last wave on the stream of its record kernels, ahead of the next file's first wave_begin_kernel; its
    // facets_end is recorded again so that ngsq_finish waits for this kernel too
    cudaStream_t st = (e->cfg.flags & NGSQ_F_SERIAL_STAGES) ? e->s_comp : e->s_scan;
    file_end_kernel<<<1, 1, 0, st>>>(e->d_state);
    CU(cudaGetLastError());
    e->other_launches++;
    CU(cudaEventRecord(e->waves.back().facets_end, st));
  }
  e->awaiting_range = true;
  return NGSQ_OK;
}

int ngsq_set_read_groups(ngsq_engine* e, uint32_t n, const char* ids, size_t ids_bytes) {
  if (!e) return NGSQ_E_ARG;
  if (!rg_on(e)) return fail(e, NGSQ_E_ARG, "ngsq_set_read_groups: the engine was created without NGSQ_F_READ_GROUPS");
  if (e->run_started) return fail(e, NGSQ_E_ARG, "ngsq_set_read_groups must precede the first submit");
  if (!e->d_res) return fail(e, NGSQ_E_ARG, "ngsq_set_read_groups: call ngsq_set_references first");
  if (n > 65534) return fail(e, NGSQ_E_ARG, "ngsq_set_read_groups: %u read groups, at most 65534", n);
  if (n && !ids) return fail(e, NGSQ_E_ARG, "ngsq_set_read_groups: ids is NULL");
  std::vector<uint32_t> off(n + 1, 0);
  std::vector<std::string> seen;
  size_t o = 0;
  for (uint32_t g = 0; g < n; ++g) {
    const void* z = o < ids_bytes ? memchr(ids + o, 0, ids_bytes - o) : nullptr;
    if (!z) return fail(e, NGSQ_E_ARG, "ngsq_set_read_groups: ids holds fewer than %u NUL-terminated IDs", n);
    const size_t len = (size_t)((const char*)z - (ids + o));
    if (!len) return fail(e, NGSQ_E_ARG, "ngsq_set_read_groups: read group %u has an empty ID", g);
    seen.emplace_back(ids + o, len);
    off[g] = (uint32_t)o;
    o += len + 1;
  }
  off[n] = (uint32_t)o;
  if (o != ids_bytes) return fail(e, NGSQ_E_ARG, "ngsq_set_read_groups: ids holds %zu bytes after its %u IDs", ids_bytes - o, n);
  std::vector<std::string> sorted = seen;
  std::sort(sorted.begin(), sorted.end());
  for (size_t i = 1; i < sorted.size(); ++i)
    if (sorted[i] == sorted[i - 1]) return fail(e, NGSQ_E_ARG, "ngsq_set_read_groups: the ID \"%s\" is given twice", sorted[i].c_str());
  // open addressing by FNV-1a, at most half full
  uint32_t slots = 2;
  while (slots < 2 * n) slots <<= 1;
  std::vector<uint32_t> table(slots, kRgEmpty);
  uint64_t sig = 0xcbf29ce484222325ull ^ n;
  for (uint32_t g = 0; g < n; ++g) {
    uint32_t s = rg_hash((const uint8_t*)ids + off[g], (uint32_t)seen[g].size()) & (slots - 1);
    while (table[s] != kRgEmpty) s = (s + 1) & (slots - 1);
    table[s] = g + 1;
  }
  for (size_t i = 0; i < ids_bytes; ++i) sig = (sig ^ (uint8_t)ids[i]) * 0x100000001b3ull;
  CU(cudaSetDevice(e->device));
  e->rg_set = false;
  e->rg_n = n;
  int rc;
  if ((rc = alloc_groups(e, e->qpos_cap, false))) return rc;
  if ((rc = fresh(e, e->d_rg_ids, std::max<size_t>(ids_bytes, 1), "read-group IDs"))) return rc;
  if ((rc = fresh(e, e->d_rg_id_off, (size_t)n + 1, "read-group IDs"))) return rc;
  if ((rc = fresh(e, e->d_rg_table, slots, "read-group table"))) return rc;
  if ((rc = fresh(e, e->d_rg_count, (size_t)n + 1, "read-group counts"))) return rc;
  if ((rc = fresh(e, e->d_rg_cursor, (size_t)n + 1, "read-group counts"))) return rc;
  if (ids_bytes) CU(cudaMemcpy(e->d_rg_ids, ids, ids_bytes, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(e->d_rg_id_off, off.data(), off.size() * 4, cudaMemcpyHostToDevice));
  CU(cudaMemcpy(e->d_rg_table, table.data(), table.size() * 4, cudaMemcpyHostToDevice));
  e->rg_mask = slots - 1;
  e->rg_sig = sig;
  e->rg_cap = 0;  // the buckets hold 32 slots of padding per group: sized again by the first wave
  e->rg_set = true;
  e->layout_agreed = false;
  return NGSQ_OK;
}

int ngsq_select_read_group(ngsq_engine* e, int32_t g) {
  if (!e) return NGSQ_E_ARG;
  if (!rg_on(e)) return fail(e, NGSQ_E_ARG, "ngsq_select_read_group: the engine was created without NGSQ_F_READ_GROUPS");
  if (!e->finished || e->h_grp_sums.empty()) return fail(e, NGSQ_E_ARG, "ngsq_select_read_group before ngsq_finish");
  if (g < -1 || g > (int32_t)e->rg_n) return fail(e, NGSQ_E_ARG, "ngsq_select_read_group: group %d outside [-1, %u]", g, e->rg_n);
  e->rg_sel = g;
  return NGSQ_OK;
}

int ngsq_progress(ngsq_engine* e, uint64_t* records) {
  if (!e || !records) return NGSQ_E_ARG;
  // waves complete in order: consume the probes of those whose scan has finished (never blocks)
  while (e->prog_seen < e->waves.size()) {
    const auto& w = e->waves[e->prog_seen];
    if (cudaEventQuery(w.scan_end) != cudaSuccess) break;
    if (w.scanned && e->waves.size() - e->prog_seen <= kProgSlots) {
      const uint64_t* p = e->h_prog + 2 * (e->prog_seen % kProgSlots);
      e->prog_records = p[0] + p[1];
    }
    e->prog_seen++;
  }
  if (e->finished) e->prog_records = e->stats.records;
  *records = e->prog_records;
  return NGSQ_OK;
}

int ngsq_wait_copied(ngsq_engine* e, uint32_t submit_index) {
  if (!e) return NGSQ_E_ARG;
  if (submit_index >= e->chunks.size()) return fail(e, NGSQ_E_ARG, "submit %u does not exist in this run (%zu so far)", submit_index, e->chunks.size());
  CU(cudaSetDevice(e->device));
  CU(cudaEventSynchronize(e->chunks[submit_index].copied));
  return NGSQ_OK;
}

int ngsq_submit_device(ngsq_engine* e, const void* dev_bgzf, size_t nbytes, const ngsq_block* blocks, uint32_t n_blocks) {
  if (!e || !dev_bgzf || (!blocks && n_blocks)) return fail(e, NGSQ_E_ARG, "bad submit arguments");
  if (e->finished) return fail(e, NGSQ_E_ARG, "submit after finish; call ngsq_reset");
  if (!e->range_set) return fail(e, NGSQ_E_ARG, "ngsq_set_range must precede the first submit");
  if (e->awaiting_range) return fail(e, NGSQ_E_ARG, "ngsq_set_range must follow ngsq_next_file before the next file's first submit");
  CU(cudaSetDevice(e->device));
  int rc = start_run(e);
  if (rc) return rc;
  if (!n_blocks) return NGSQ_OK;
  const ngsq_block& last = blocks[n_blocks - 1];
  if (last.coffset + last.csize - blocks[0].coffset > nbytes) return fail(e, NGSQ_E_TRUNCATED, "block table runs past the device buffer");
  e->comp_bytes_total += nbytes;
  const uint32_t first_new = (uint32_t)e->h_blocks.size();
  rc = append_blocks(e, blocks, n_blocks, (uint64_t)(uintptr_t)dev_bgzf, blocks[0].coffset);
  if (rc) return rc;
  rc = upload_descriptors(e, first_new, (uint32_t)e->h_blocks.size());
  if (rc) return rc;
  cudaEvent_t ev;
  CU(cudaEventCreateWithFlags(&ev, e->trace ? cudaEventDefault : cudaEventDisableTiming));
  CU(cudaEventRecord(ev, e->s_copy));
  e->chunks.push_back({ev, (uint32_t)e->h_blocks.size()});
  // resident data: every wave is enqueued at once (the caller's buffer is used in place)
  return launch_pending(e, (uint32_t)e->h_blocks.size(), false);
}

int ngsq_finish(ngsq_engine* e) {
  if (!e) return NGSQ_E_ARG;
  if (e->finished) return NGSQ_OK;
  CU(cudaSetDevice(e->device));
  int rc = start_run(e);
  if (rc) return rc;
  const uint32_t nb = (uint32_t)e->h_blocks.size();
  if (nb && !e->range_set) return fail(e, NGSQ_E_ARG, "ngsq_set_range was not called");
  rc = launch_pending(e, nb, true);
  if (rc) return rc;
  if (nb > e->file_b0) {
    // a virtual offset behind the last block can only mean "end of data"
    if (!e->start_resolved && (e->first_voff & 0xFFFF)) return fail(e, NGSQ_E_ARG, "virtual offset %llu is beyond the submitted data", (unsigned long long)e->first_voff);
    if (e->end_voff && !e->end_resolved && (e->end_voff & 0xFFFF)) return fail(e, NGSQ_E_ARG, "virtual offset %llu is beyond the submitted data", (unsigned long long)e->end_voff);
  }
  cudaStream_t s = e->s_comp;
  if (!e->waves.empty()) {
    int crc_rc = launch_crc(e, e->waves.back(), nullptr);
    if (crc_rc) return crc_rc;
    CU(cudaStreamWaitEvent(s, e->waves.back().facets_end, 0));  // the scan stream's last kernel
  }
  CU(cudaEventRecord(e->ev_d, s));
  // K9 (split references wait for the merge: their arrays hold this shard's part only)
  if (e->cfg.flags & NGSQ_F_COVERAGE) {
    for (uint32_t c = 0; c < e->n_ref; ++c)
      if (e->cov_enabled[c] && !e->split_ref[c]) launch_cov_resolve(e, c, s);
    CU(cudaGetLastError());
  }
  CU(cudaEventRecord(e->ev_e, s));
  // K11 teardown (edits.rs:318-334): the VAF histogram over the per-position counters of every wave; with split references,
  // one launch per run of contiguous non-split contigs (the counters are laid out contig after contig)
  const bool do_edits = edits_loaded(e);
  if (do_edits && e->ed_pos_total && !e->waves.empty()) {
    if (!e->n_split) {
      launch_vaf(e, 0, e->ed_pos_total, s);
    } else {
      uint64_t run_beg = 0, run_end = 0;
      for (uint32_t c = 0; c <= e->n_ref; ++c) {
        if (c < e->n_ref && !e->split_ref[c]) { run_end = e->ed_contigs[c].pos_off + e->ed_contigs[c].hdr_len + 1; continue; }
        if (run_end > run_beg) launch_vaf(e, run_beg, run_end - run_beg, s);
        if (c < e->n_ref) run_beg = run_end = e->ed_contigs[c].pos_off + e->ed_contigs[c].hdr_len + 1;
      }
    }
    CU(cudaGetLastError());
  }
  if (do_edits) {
    e->h_ed_res.resize(E_WORDS);
    CU(cudaMemcpyAsync(e->h_ed_res.data(), e->d_ed_res, E_WORDS * 8, cudaMemcpyDeviceToHost, s));
  }
  const bool do_features = (e->cfg.flags & NGSQ_F_FEATURES) && e->d_ft_res && e->ft_model_set && e->ft_contigs.size() == e->n_ref;
  if ((e->cfg.flags & NGSQ_F_FEATURES) && !do_features) return fail(e, NGSQ_E_ARG, "NGSQ_F_FEATURES needs ngsq_set_feature_model before the first submit");
  if (do_features) {
    e->h_ft_res.resize(F_WORDS);
    CU(cudaMemcpyAsync(e->h_ft_res.data(), e->d_ft_res, F_WORDS * 8, cudaMemcpyDeviceToHost, s));
  }
  CU(cudaEventRecord(e->ev_g, s));
  // the step ends when the CRC stream is done too (its last event closes the device-timed region)
  if (!e->waves.empty()) CU(cudaStreamWaitEvent(s, e->waves.back().crc_end, 0));
  CU(cudaMemcpyAsync(e->h_state, e->d_state, sizeof(RunState), cudaMemcpyDeviceToHost, s));
  // results: everything but the quality table now, the table's rows once their number is known
  e->h_res.assign(e->qual_off, 0);
  CU(cudaMemcpyAsync(e->h_res.data(), e->d_res, (size_t)e->qual_off * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  const uint32_t qpos = (uint32_t)std::min<uint64_t>(e->h_res[R_QUAL_POSITIONS], e->qpos_cap);
  e->h_res.resize((size_t)e->qual_off + (size_t)qpos * 94);
  if (qpos) CU(cudaMemcpyAsync(e->h_res.data() + e->qual_off, e->d_res + e->qual_off, (size_t)qpos * 94 * 8, cudaMemcpyDeviceToHost, s));
  if (rg_on(e)) {
    int grc = fetch_groups(e, s);
    if (grc) return grc;
  }
  CU(cudaEventRecord(e->ev_f, s));
  CU(cudaStreamSynchronize(s));
  e->finished = true;
  if (rg_on(e)) e->grp_dirty = std::min(e->grp_rows, std::max<uint32_t>(e->h_state->max_lseq, 256));
  e->h_qpos = qpos;
  e->qpos_dirty = std::max(e->qpos_dirty, std::min<uint32_t>(std::max<uint32_t>(e->h_state->max_lseq, qpos), e->qpos_cap));
  // stats
  const RunState& R = *e->h_state;
  ngsq_stats& st = e->stats;
  st.records = R.rec_base + R.wave_rec; st.blocks = nb; st.compressed_bytes = e->comp_bytes_total; st.inflated_bytes = e->out_used; st.max_read_len = R.max_lseq;
  st.ms_inflate = st.ms_inflate_decode = st.ms_inflate_resolve = st.ms_crc = st.ms_scan = st.ms_facets = 0;
  for (auto& p : e->waves) {
    float ms = 0;
    cudaEventElapsedTime(&ms, p.begin, p.resolved); st.ms_inflate += ms;
    cudaEventElapsedTime(&ms, p.decoded_from, p.decoded); st.ms_inflate_decode += ms;
    cudaEventElapsedTime(&ms, p.decoded, p.resolved); st.ms_inflate_resolve += ms;
    cudaEventElapsedTime(&ms, p.crc_begin, p.crc_end); st.ms_crc += ms;
    cudaEventElapsedTime(&ms, p.scan_begin, p.scan_end); st.ms_scan += ms;
    cudaEventElapsedTime(&ms, p.scan_end, p.facets_end); st.ms_facets += ms;
  }
  cudaEventElapsedTime(&st.ms_coverage, e->ev_d, e->ev_e);
  cudaEventElapsedTime(&st.ms_edits, e->ev_e, e->ev_g);
  cudaEventElapsedTime(&st.ms_total, e->ev_start, e->ev_f);
  if (!e->waves.empty()) cudaEventElapsedTime(&st.ms_tail, e->waves.back().begin, e->ev_f);
  st.waves = (uint32_t)e->waves.size();
  st.other_launches = e->other_launches;
  if (e->trace) {
    auto at = [&](cudaEvent_t ev) { float ms = 0; cudaEventElapsedTime(&ms, e->ev_start, ev); return ms; };
    fprintf(stderr, "[ngsq trace] %zu chunks, %zu waves, total %.1f ms (ms since the first submit)\n", e->chunks.size(), e->waves.size(), st.ms_total);
    for (size_t i = 0; i < e->chunks.size(); ++i)
      if (i % 8 == 7 || i + 1 == e->chunks.size()) fprintf(stderr, "[ngsq trace] chunk %3zu copied at %8.1f (blocks < %u)\n", i, at(e->chunks[i].copied), e->chunks[i].blocks_end);
    for (size_t i = 0; i < e->waves.size(); ++i) {
      const auto& w = e->waves[i];
      fprintf(stderr, "[ngsq trace] wave %2zu blocks<%7u host %7.1f | begin %7.1f decode %7.1f..%7.1f resolved %7.1f | scan %7.1f..%7.1f facets %7.1f | crc %7.1f..%7.1f\n", i, w.b1,
              i < e->host_ms.size() ? e->host_ms[i] : -1.0, at(w.begin), at(w.decoded_from), at(w.decoded), at(w.resolved), at(w.scan_begin), at(w.scan_end), at(w.facets_end), at(w.crc_begin), at(w.crc_end));
    }
    fprintf(stderr, "[ngsq trace] coverage %.1f..%.1f end %.1f\n", at(e->ev_d), at(e->ev_e), at(e->ev_f));
    if (rg_on(e)) fprintf(stderr, "[ngsq trace] rg_facets_kernel: %d CTAs per SM, %zu bytes of shared memory each\n", e->rg_occ, e->rg_smem);
  }
  // verdicts, in the order the reference would meet them: a block that does not inflate, a block whose CRC32 is wrong
  // (its garbage bytes break the record chain too: CRC first), then the record chain, then the records
  if (R.fatal & kFatalInflate) {
    const uint64_t b = R.bad_block >> 8;
    const uint32_t code = (uint32_t)(R.bad_block & 0xFF);
    return fail(e, NGSQ_E_BAD_BLOCK, "BGZF block at file offset %llu failed to inflate (%s)", (unsigned long long)(b < nb ? e->h_blocks[b].coff : 0),
                code == kBlkIsize ? "ISIZE mismatch" : code == kBlkOverrun ? "output overrun / bad distance" : "invalid DEFLATE stream");
  }
  if (R.crc_bad) return fail(e, NGSQ_E_CRC, "%u BGZF block(s) failed the CRC32 check", R.crc_bad);
  if ((R.fatal & kFatalTruncated) || (!R.fatal && R.cn_len && !R.end_pending && !R.end_reached))
    return fail(e, NGSQ_E_TRUNCATED, "record chain runs past the end of the submitted data");
  if (R.fatal & kFatalBadRecord) return fail(e, NGSQ_E_BAD_RECORD, "malformed record length on the record chain");
  if (R.fatal & kFatalChain) return fail(e, NGSQ_E_CHAIN, "record chain does not close on the shard's end offset");
  if (R.fatal & kFatalCarry)
    return fail(e, NGSQ_E_BAD_RECORD, "a record is longer than the %u bytes the engine carries between two waves (raise ngsq_config.carry_bytes)", e->headroom);
  if (R.fatal & kFatalRecTable) return fail(e, NGSQ_E_CHAIN, "record table overflow");
  if (e->h_res[R_ERR_QUAL]) return fail(e, NGSQ_E_QUAL_RANGE, "a record holds a quality score above 93 (the reference's decoder rejects it)");
  if (e->h_res[R_ERR_RECORD]) return fail(e, NGSQ_E_BAD_RECORD, "malformed BAM record (field overrun, CIGAR op > 8, reference id out of range, or a mapped pair without reference ids)");
  if (R.qual_overflow)
    return fail(e, NGSQ_E_QUAL_CAP, "a read of %u bases exceeds the %u positions of the quality table: call ngsq_set_quality_positions(%u) (or set ngsq_config.quality_positions) and run again",
                R.qual_overflow, e->qpos_cap, R.qual_overflow);
  if (do_edits && e->h_ed_res[E_ERR]) {
    static const char* const kinds[] = {"", "", "Could not parse read name", "sequence not found in reference FASTA", "record reaches past the end of the reference sequence",
                                        "invalid base in the reference sequence", "step-through: no reference base left", "step-through: no record base left",
                                        "step-through: reference sequence was not fully consumed", "step-through: record sequence was not fully consumed",
                                        "more than 512 edits in one read", "matched position beyond the sequence length of the header", "invalid CIGAR operation"};
    const uint64_t k = e->h_ed_res[E_ERR];
    return fail(e, NGSQ_E_EDITS, "Edits: %s (the reference aborts the run here)", k < sizeof kinds / sizeof *kinds ? kinds[k] : "unknown failure");
  }
  if (do_features && e->h_ft_res[F_ERR]) {
    static const char* const kinds[] = {"", "Could not parse read name", "Could not parse reference sequence id for read", "Could not parse record's start position.",
                                        "invalid CIGAR operation"};
    const uint64_t k = e->h_ft_res[F_ERR];
    return fail(e, NGSQ_E_FEATURES, "Genomic Features: %s (the reference aborts the run here)", k < sizeof kinds / sizeof *kinds ? kinds[k] : "unknown failure");
  }
  if (ix_on(e)) return finish_index(e);
  return NGSQ_OK;
}

namespace {
// ngsq_get_bai (csi = false) and ngsq_get_csi: the index bytes of a finished NGSQ_F_INDEX engine of that format
int get_index(ngsq_engine* e, bool csi, uint8_t* out, size_t cap, size_t* n_out) {
  if (!e) return NGSQ_E_ARG;
  const char* fn = csi ? "ngsq_get_csi" : "ngsq_get_bai";
  if (e->cfg.flags & NGSQ_F_INDEX_PART)
    return fail(e, NGSQ_E_ARG, "%s: this engine indexed one part of a file (NGSQ_F_INDEX_PART); join the finished parts with %s", fn,
                ix_csi(e) ? "ngsq_join_csi" : "ngsq_join_bai");
  if (!(e->cfg.flags & NGSQ_F_INDEX)) return fail(e, NGSQ_E_ARG, "%s: the engine was created without NGSQ_F_INDEX", fn);
  if (csi && !ix_csi(e)) return fail(e, NGSQ_E_ARG, "ngsq_get_csi: the engine builds a BAI (created without NGSQ_F_INDEX_CSI); read it with ngsq_get_bai");
  if (!csi && ix_csi(e)) return fail(e, NGSQ_E_ARG, "ngsq_get_bai: the engine builds a CSI (NGSQ_F_INDEX_CSI); read it with ngsq_get_csi");
  if (!e->finished || e->ix_bytes.empty()) return fail(e, NGSQ_E_ARG, "%s: no index before a successful ngsq_finish", fn);
  if (n_out) *n_out = e->ix_bytes.size();
  if (!out && !cap) return NGSQ_OK;
  if (!out || cap < e->ix_bytes.size()) return fail(e, NGSQ_E_ARG, "%s: buffer holds %zu bytes, %zu needed", fn, cap, e->ix_bytes.size());
  memcpy(out, e->ix_bytes.data(), e->ix_bytes.size());
  return NGSQ_OK;
}
}  // namespace

int ngsq_get_bai(ngsq_engine* e, uint8_t* out, size_t cap, size_t* n_out) { return get_index(e, false, out, cap, n_out); }
int ngsq_get_csi(ngsq_engine* e, uint8_t* out, size_t cap, size_t* n_out) { return get_index(e, true, out, cap, n_out); }

int ngsq_set_index_binning(ngsq_engine* e, uint32_t min_shift, uint32_t depth) {
  if (!e) return NGSQ_E_ARG;
  if (!ix_on(e) || !ix_csi(e)) return fail(e, NGSQ_E_ARG, "ngsq_set_index_binning: the engine was created without NGSQ_F_INDEX_CSI");
  if (e->d_ref_len) return fail(e, NGSQ_E_ARG, "ngsq_set_index_binning must precede ngsq_set_references (the window tables depend on it)");
  if (min_shift < kCsiMinShiftLo || min_shift > kCsiMinShiftHi)
    return fail(e, NGSQ_E_ARG, "ngsq_set_index_binning: min_shift %u is outside [%u, %u]", min_shift, kCsiMinShiftLo, kCsiMinShiftHi);
  if (depth > kCsiDepthHi) return fail(e, NGSQ_E_ARG, "ngsq_set_index_binning: depth %u is outside [1, %u] (0 = the default rule)", depth, kCsiDepthHi);
  e->ix_min_shift = min_shift;
  e->ix_depth_req = depth;
  return NGSQ_OK;
}

// the sample's counters, or those of the selected read group (same offsets)
#define RESULT_WORDS() (e->rg_sel >= 0 ? &e->h_grp_sums[(size_t)e->rg_sel * kGroupSums] : e->h_res.data())
#define SAMPLE_ONLY(what)                                                                \
  if (e && e->rg_sel >= 0) return fail(e, NGSQ_E_ARG, "%s: read group %d is selected, and this facet is the sample's only (ngsq_select_read_group(e, -1))", what, e->rg_sel)

int ngsq_get_features(ngsq_engine* e, uint64_t counts[9]) {
  if (!e || !counts) return NGSQ_E_ARG;
  SAMPLE_ONLY("ngsq_get_features");
  if (!e->finished || e->h_ft_res.size() != F_WORDS) return fail(e, NGSQ_E_ARG, "Genomic Features results requested before ngsq_finish or without NGSQ_F_FEATURES");
  if (e->h_ft_res[F_ERR]) return fail(e, NGSQ_E_FEATURES, "the Genomic Features facet failed; no results");
  memcpy(counts, e->h_ft_res.data(), 9 * 8);
  return NGSQ_OK;
}

int ngsq_get_edits(ngsq_engine* e, uint64_t read_one[513], uint64_t read_two[513], uint64_t vaf[101], uint64_t* records) {
  if (!e) return NGSQ_E_ARG;
  SAMPLE_ONLY("ngsq_get_edits");
  if (!e->finished || e->h_ed_res.size() != E_WORDS) return fail(e, NGSQ_E_ARG, "Edits results requested before ngsq_finish or without NGSQ_F_EDITS");
  if (e->h_ed_res[E_ERR]) return fail(e, NGSQ_E_EDITS, "the Edits facet failed; no results");
  if (e->n_split && !e->split_merged)
    return fail(e, NGSQ_E_ARG, "Edits results requested before the split references were merged (ngsq_reduce or ngsq_resolve_split): the VAF histogram is incomplete");
  if (read_one) memcpy(read_one, &e->h_ed_res[E_READ_ONE], 513 * 8);
  if (read_two) memcpy(read_two, &e->h_ed_res[E_READ_TWO], 513 * 8);
  if (vaf) memcpy(vaf, &e->h_ed_res[E_VAF], 101 * 8);
  if (records) *records = e->h_ed_res[E_RECORDS];
  return NGSQ_OK;
}

// Per-position counters of one header sequence for the VAF file (edits.rs:317-340): a plain read-back, positions are
// 1-based like alignment_start + reference_ptr (edits.rs:279-281), entry 0 is never written.
int ngsq_get_edit_positions(ngsq_engine* e, uint32_t ref, uint32_t* refs, uint32_t* alts, uint64_t n) {
  if (!e) return NGSQ_E_ARG;
  SAMPLE_ONLY("ngsq_get_edit_positions");
  if (!e->finished || e->h_ed_res.size() != E_WORDS) return fail(e, NGSQ_E_ARG, "Edits results requested before ngsq_finish or without NGSQ_F_EDITS");
  if (e->h_ed_res[E_ERR]) return fail(e, NGSQ_E_EDITS, "the Edits facet failed; no results");
  if (ref >= e->n_ref || ref >= e->ed_contigs.size() || !refs || !alts) return fail(e, NGSQ_E_ARG, "ngsq_get_edit_positions: bad reference id or null output");
  if (is_split(e, ref) && !e->split_merged)
    return fail(e, NGSQ_E_ARG, "ngsq_get_edit_positions: reference %u is split between shards and not merged yet (ngsq_reduce or ngsq_resolve_split)", ref);
  const EditsContig& c = e->ed_contigs[ref];
  if (n != (uint64_t)c.hdr_len + 1) return fail(e, NGSQ_E_ARG, "ngsq_get_edit_positions: reference %u has %u + 1 positions, %llu requested", ref, c.hdr_len, (unsigned long long)n);
  CU(cudaSetDevice(e->device));
  CU(cudaMemcpy(refs, e->d_ed_refs + c.pos_off, n * 4, cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(alts, e->d_ed_alts + c.pos_off, n * 4, cudaMemcpyDeviceToHost));
  return NGSQ_OK;
}

#define NEED_RESULTS()                                                                   \
  if (!e) return NGSQ_E_ARG;                                                             \
  if (!e->finished || e->h_res.empty()) return fail(e, NGSQ_E_ARG, "results requested before ngsq_finish")

int ngsq_get_general(ngsq_engine* e, uint64_t out[34]) {
  NEED_RESULTS();
  memcpy(out, RESULT_WORDS() + R_GENERAL, 34 * 8);
  return NGSQ_OK;
}

int ngsq_get_tlen(ngsq_engine* e, uint64_t hist[1025], uint64_t* processed, uint64_t* ignored) {
  NEED_RESULTS();
  const uint64_t* w = RESULT_WORDS();
  memcpy(hist, w + R_TLEN_HIST, 1025 * 8);
  *processed = w[R_TLEN_PROCESSED];
  *ignored = w[R_TLEN_IGNORED];
  return NGSQ_OK;
}

int ngsq_get_gc(ngsq_engine* e, uint64_t hist[101], uint64_t nuc[3], uint64_t rec[3]) {
  NEED_RESULTS();
  const uint64_t* w = RESULT_WORDS();
  memcpy(hist, w + R_GC_HIST, 101 * 8);
  memcpy(nuc, w + R_GC_NUC, 24);
  memcpy(rec, w + R_GC_REC, 24);
  return NGSQ_OK;
}

int ngsq_get_quality(ngsq_engine* e, uint64_t* out, size_t cap_positions, uint32_t* n_positions) {
  NEED_RESULTS();
  const bool grp = e->rg_sel >= 0;
  uint32_t n = grp ? (uint32_t)e->h_grp_qlen[e->rg_sel] : e->h_qpos;
  if (n_positions) *n_positions = n;
  if (!out) return NGSQ_OK;
  if (cap_positions < n) return fail(e, NGSQ_E_ARG, "quality buffer holds %zu positions, %u needed", cap_positions, n);
  memcpy(out, grp ? e->h_grp_qual[e->rg_sel].data() : &e->h_res[e->qual_off], (size_t)n * 94 * 8);
  return NGSQ_OK;
}

int ngsq_get_coverage_contig(ngsq_engine* e, uint32_t ref, ngsq_cov_ints* out, uint64_t* bin_sums, size_t cap) {
  NEED_RESULTS();
  SAMPLE_ONLY("ngsq_get_coverage_contig");
  if (ref >= e->n_ref || !out) return fail(e, NGSQ_E_ARG, "bad reference index");
  if (is_split(e, ref) && !e->split_merged)
    return fail(e, NGSQ_E_ARG, "reference %u is split between shards and not merged yet (ngsq_reduce or ngsq_resolve_split)", ref);
  memset(out, 0, sizeof *out);
  if (!e->cov_enabled[ref]) return NGSQ_OK;
  const uint64_t* slot = &e->h_res[e->cov_slot[ref]];
  out->touched = slot[COV_TOUCHED] ? 1 : 0;
  if (!out->touched) return NGSQ_OK;
  out->n_bins = e->cov_nbins[ref];
  out->pileup_too_large = slot[COV_TOO_LARGE];
  memcpy(out->hist, slot + COV_HIST, 2049 * 8);
  if (bin_sums) {
    if (cap < out->n_bins) return fail(e, NGSQ_E_ARG, "bin buffer holds %zu entries, %u needed", cap, out->n_bins);
    memcpy(bin_sums, slot + COV_BINS, (size_t)out->n_bins * 8);
  }
  return NGSQ_OK;
}

int ngsq_get_coverage_global(ngsq_engine* e, uint64_t* nonsensical_records) {
  NEED_RESULTS();
  SAMPLE_ONLY("ngsq_get_coverage_global");
  *nonsensical_records = e->h_res[R_NONSENSICAL];
  return NGSQ_OK;
}

int ngsq_get_stats(ngsq_engine* e, ngsq_stats* out) {
  if (!e || !out) return NGSQ_E_ARG;
  *out = e->stats;
  return NGSQ_OK;
}

int ngsq_nccl_unique_id(char out[128]) {
  std::string err;
  if (!load_nccl(err)) { g_create_err = err; return NGSQ_E_NCCL; }
  NcclId id;
  int rc = g_nccl.GetUniqueId(&id);
  if (rc) { g_create_err = std::string("ncclGetUniqueId: ") + (g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"); return NGSQ_E_NCCL; }
  memcpy(out, id.b, 128);
  return NGSQ_OK;
}

int ngsq_comm_init(ngsq_engine* e, int n_ranks, int rank, const char id[128]) {
  if (!e || !id) return NGSQ_E_ARG;
  std::string err;
  if (!load_nccl(err)) return fail(e, NGSQ_E_NCCL, "%s", err.c_str());
  CU(cudaSetDevice(e->device));
  // ncclCommInitRank(ncclComm_t*, int, ncclUniqueId /*by value*/, int)
  typedef int (*init_fn)(void**, int, NcclId, int);
  NcclId nid;
  memcpy(nid.b, id, 128);
  int rc = ((init_fn)g_nccl.CommInitRank)(&e->comm, n_ranks, nid, rank);
  if (rc) return fail(e, NGSQ_E_NCCL, "ncclCommInitRank: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
  e->n_ranks = n_ranks;
  e->rank = rank;
  return NGSQ_OK;
}

int ngsq_set_quality_positions(ngsq_engine* e, uint32_t n_positions) {
  if (!e) return NGSQ_E_ARG;
  if (e->run_started && !e->finished) return fail(e, NGSQ_E_ARG, "ngsq_set_quality_positions: a run is in flight");
  CU(cudaSetDevice(e->device));
  e->cfg.quality_positions = std::max(e->cfg.quality_positions, n_positions);
  if (!e->d_cov_slot && !e->n_ref) return NGSQ_OK;  // no layout yet: ngsq_set_references will size the table
  return ensure_res(e, n_positions, true);
}

int ngsq_result_buffer(ngsq_engine* e, void** dev_ptr, size_t* n_words) {
  if (!e || !dev_ptr || !n_words) return NGSQ_E_ARG;
  *dev_ptr = e->d_res;
  *n_words = e->res_words;
  return NGSQ_OK;
}

// After an external reduction of the device buffer, refresh the host copy.
int ngsq_refresh_results(ngsq_engine* e) {
  if (!e || !e->finished) return fail(e, NGSQ_E_ARG, "refresh before finish");
  CU(cudaSetDevice(e->device));
  cudaStream_t s = e->s_comp;
  e->h_res.assign(e->qual_off, 0);
  CU(cudaMemcpyAsync(e->h_res.data(), e->d_res, (size_t)e->qual_off * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  const uint32_t qpos = (uint32_t)std::min<uint64_t>(e->h_res[R_QUAL_POSITIONS], e->qpos_cap);
  e->h_res.resize((size_t)e->qual_off + (size_t)qpos * 94);
  if (qpos) CU(cudaMemcpyAsync(e->h_res.data() + e->qual_off, e->d_res + e->qual_off, (size_t)qpos * 94 * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  e->h_qpos = qpos;
  e->qpos_dirty = std::max(e->qpos_dirty, qpos);
  return NGSQ_OK;
}

// K10.  ONE sum collective in the steady state: every rank parks its own quality length and layout word in its slot of
// the fixed part (all other ranks hold zeros there), so the all-reduce also hands every rank the max over ranks and the
// proof that the layouts agree.  Reads longer than kReduceQualRows need a second call for the rest of the table; the very
// first reduce of an engine agrees on the layout beforehand (a mismatch would mean mismatched counts inside NCCL).
int ngsq_reduce(ngsq_engine* e, int root) {
  if (!e || !e->finished) return fail(e, NGSQ_E_ARG, "reduce before finish");
  if (e->cfg.flags & NGSQ_F_INDEX) return fail(e, NGSQ_E_ARG, "ngsq_reduce: an index is built by one engine over the whole file (NGSQ_F_INDEX)");
  if (!e->comm) return fail(e, NGSQ_E_NCCL, "ngsq_comm_init was not called");
  if (e->n_ranks > (int)kMaxRanks) return fail(e, NGSQ_E_ARG, "at most %u ranks", kMaxRanks);
  CU(cudaSetDevice(e->device));
  cudaStream_t s = e->s_comp;
  CU(cudaEventRecord(e->ev_a, s));
  const int ncclInt32 = 2, ncclUint32 = 3, ncclUint64 = 5, ncclSum = 0, ncclMax = 2;
  auto nccl_err = [&](const char* what, int rc) { return fail(e, NGSQ_E_NCCL, "%s: %s", what, g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?"); };
  // the split set is part of the agreed layout: ranks that disagree on it would issue different collectives below
  const uint64_t layout = ((uint64_t)e->qual_off | ((uint64_t)e->qpos_cap << 32)) ^ split_signature(e) ^
                          (rg_on(e) ? e->rg_sig * 31 + e->grp_rows : 0);
  int rc;
  if (!e->layout_agreed) {
    uint64_t agree[2] = {layout, ~layout};
    uint64_t* d_agree = e->d_res + R_RANK_LAYOUT;  // scratch: rewritten below
    CU(cudaMemcpyAsync(d_agree, agree, sizeof agree, cudaMemcpyHostToDevice, s));
    rc = g_nccl.AllReduce(d_agree, d_agree, 2, ncclUint64, ncclMax, e->comm, s);
    if (rc) return nccl_err("ncclAllReduce", rc);
    CU(cudaMemcpyAsync(agree, d_agree, sizeof agree, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    if (agree[0] != layout || ~agree[1] != layout)
      return fail(e, NGSQ_E_ARG, "result layouts differ across ranks: ngsq_set_references must get the same lengths and coverage mask, ngsq_split_reference the same references, and ngsq_config.quality_positions the same value, on every rank");
    e->layout_agreed = true;
    e->other_launches += 1;
  }
  // split references first: every rank's partial arrays summed onto the root, which resolves them before the result buffer
  // (its slots of those contigs included) is summed below
  if (e->n_split && !e->split_merged) {
    const bool edits = edits_loaded(e) && e->ed_pos_total;
    for (uint32_t c = 0; c < e->n_ref; ++c) {
      if (!e->split_ref[c]) continue;
      if (e->cov_enabled[c]) {
        int32_t* df = e->d_diff + e->diff_base[c];
        int32_t* ts = e->d_tile_sum + e->tile_off[c];
        uint64_t* touched = e->d_res + e->cov_slot[c] + COV_TOUCHED;
        if ((rc = g_nccl.Reduce(df, df, (size_t)e->ref_len[c] + 2, ncclInt32, ncclSum, root, e->comm, s))) return nccl_err("ncclReduce (split coverage)", rc);
        if ((rc = g_nccl.Reduce(ts, ts, cov_tiles(e, c), ncclInt32, ncclSum, root, e->comm, s))) return nccl_err("ncclReduce (split tile sums)", rc);
        if ((rc = g_nccl.Reduce(touched, touched, 1, ncclUint64, ncclSum, root, e->comm, s))) return nccl_err("ncclReduce (split touched)", rc);
        e->other_launches += 3;
      }
      if (edits) {
        const EditsContig& ec = e->ed_contigs[c];
        const size_t n = (size_t)ec.hdr_len + 1;
        if ((rc = g_nccl.Reduce(e->d_ed_refs + ec.pos_off, e->d_ed_refs + ec.pos_off, n, ncclUint32, ncclSum, root, e->comm, s))) return nccl_err("ncclReduce (split edits)", rc);
        if ((rc = g_nccl.Reduce(e->d_ed_alts + ec.pos_off, e->d_ed_alts + ec.pos_off, n, ncclUint32, ncclSum, root, e->comm, s))) return nccl_err("ncclReduce (split edits)", rc);
        e->other_launches += 2;
      }
    }
    rc = merge_split_local(e, e->rank == root, s);
    if (rc) return rc;
  }
  std::vector<uint64_t> slots(2 * kMaxRanks + 0, 0);
  slots[e->rank] = e->h_qpos;
  slots[kMaxRanks + e->rank] = layout;
  CU(cudaMemcpyAsync(e->d_res + R_RANK_QPOS, slots.data(), slots.size() * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemsetAsync(e->d_res + R_QUAL_POSITIONS, 0, 8, s));  // a max, not a sum: rebuilt from the slots
  const uint32_t rows1 = std::min<uint32_t>(kReduceQualRows, e->qpos_cap);
  const size_t n1 = (size_t)e->qual_off + (size_t)rows1 * 94;
  rc = g_nccl.AllReduce(e->d_res, e->d_res, n1, ncclUint64, ncclSum, e->comm, s);
  if (rc) return nccl_err("ncclAllReduce", rc);
  CU(cudaMemcpyAsync(slots.data(), e->d_res + R_RANK_QPOS, slots.size() * 8, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  e->other_launches += 1;
  uint64_t qmax = 0;
  for (int r = 0; r < e->n_ranks; ++r) {
    qmax = std::max(qmax, slots[r]);
    if (slots[kMaxRanks + r] != layout) return fail(e, NGSQ_E_ARG, "result layouts differ across ranks (rank %d)", r);
  }
  if (qmax > rows1) {  // long reads: the rest of the table (every rank knows qmax now)
    const size_t n2 = (size_t)(std::min<uint64_t>(qmax, e->qpos_cap) - rows1) * 94;
    uint64_t* rest = e->d_res + n1;
    rc = g_nccl.Reduce(rest, rest, n2, ncclUint64, ncclSum, root, e->comm, s);
    if (rc) return nccl_err("ncclReduce", rc);
    e->other_launches += 1;
  }
  CU(cudaMemcpyAsync(e->d_res + R_QUAL_POSITIONS, &qmax, 8, cudaMemcpyHostToDevice, s));
  CU(cudaStreamSynchronize(s));
  if ((e->cfg.flags & NGSQ_F_EDITS) && e->d_ed_res && e->h_ed_res.size() == E_WORDS) {
    // additive like everything else: every shard owns whole contigs, so per-position counters never meet
    rc = g_nccl.Reduce(e->d_ed_res, e->d_ed_res, E_WORDS, ncclUint64, ncclSum, root, e->comm, s);
    if (rc) return nccl_err("ncclReduce (edits)", rc);
    CU(cudaMemcpyAsync(e->h_ed_res.data(), e->d_ed_res, E_WORDS * 8, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    e->other_launches += 1;
  }
  if ((e->cfg.flags & NGSQ_F_FEATURES) && e->d_ft_res && e->h_ft_res.size() == F_WORDS) {
    rc = g_nccl.Reduce(e->d_ft_res, e->d_ft_res, F_WORDS, ncclUint64, ncclSum, root, e->comm, s);
    if (rc) return nccl_err("ncclReduce (features)", rc);
    CU(cudaMemcpyAsync(e->h_ft_res.data(), e->d_ft_res, F_WORDS * 8, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    e->other_launches += 1;
  }
  if (rg_on(e) && e->rg_set) {
    // the groups: lengths with max (every rank then issues the same quality reduces), counters with sum, the tables' rows
    // up to each group's length onto the root
    const uint64_t ng = (uint64_t)e->rg_n + 1, head = ng * (kGroupSums + 1);
    uint64_t* qlen = e->d_grp + ng * kGroupSums;
    if ((rc = g_nccl.AllReduce(qlen, qlen, ng, ncclUint64, ncclMax, e->comm, s))) return nccl_err("ncclAllReduce (read-group lengths)", rc);
    if ((rc = g_nccl.AllReduce(e->d_grp, e->d_grp, ng * kGroupSums, ncclUint64, ncclSum, e->comm, s))) return nccl_err("ncclAllReduce (read groups)", rc);
    std::vector<uint64_t> len(ng);
    CU(cudaMemcpyAsync(len.data(), qlen, ng * 8, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    e->other_launches += 2;
    for (uint64_t g = 0; g < ng; ++g) {
      const uint64_t rows = std::min<uint64_t>(len[g], e->grp_rows);
      if (!rows) continue;
      uint64_t* t = e->d_grp + head + g * e->grp_rows * 94;
      if ((rc = g_nccl.Reduce(t, t, rows * 94, ncclUint64, ncclSum, root, e->comm, s))) return nccl_err("ncclReduce (read-group quality)", rc);
      e->other_launches += 1;
    }
    if ((rc = fetch_groups(e, s))) return rc;
  }
  rc = ngsq_refresh_results(e);
  if (rc) return rc;
  e->split_merged = true;
  // the `touched` flags were summed: a contig two ranks scattered into would get a depth histogram that is the sum of two
  // partial resolves, not the histogram of the summed depth (shards must be contig-exclusive unless the contig was declared
  // with ngsq_split_reference, SURVEY 8(e))
  for (uint32_t c = 0; c < e->n_ref; ++c)
    if (e->cov_enabled[c] && !e->split_ref[c] && e->h_res[e->cov_slot[c] + COV_TOUCHED] > 1)
      return fail(e, NGSQ_E_ARG, "reference %u holds coverage from %llu ranks: every contig must lie in one shard", c, (unsigned long long)e->h_res[e->cov_slot[c] + COV_TOUCHED]);
  CU(cudaEventRecord(e->ev_b, s));
  CU(cudaEventSynchronize(e->ev_b));
  cudaEventElapsedTime(&e->stats.ms_reduce, e->ev_a, e->ev_b);
  e->stats.other_launches = e->other_launches;
  // touched flags were summed: any non-zero means touched (getters test != 0)
  return NGSQ_OK;
}

int ngsq_split_reference(ngsq_engine* e, uint32_t ref) {
  if (!e) return NGSQ_E_ARG;
  if (e->cfg.flags & NGSQ_F_INDEX) return fail(e, NGSQ_E_ARG, "ngsq_split_reference: an index is built by one engine over the whole file (NGSQ_F_INDEX)");
  if (e->cfg.max_records) return fail(e, NGSQ_E_ARG, "ngsq_split_reference: max_records counts records in file order on one engine");
  if (ref >= e->n_ref || e->split_ref.size() != e->n_ref) return fail(e, NGSQ_E_ARG, "ngsq_split_reference: reference %u is not in the header given to ngsq_set_references", ref);
  if (e->run_started) return fail(e, NGSQ_E_ARG, "ngsq_split_reference must precede the first submit");
  if (!e->split_ref[ref]) {
    e->split_ref[ref] = 1;
    ++e->n_split;
    e->layout_agreed = false;
  }
  return NGSQ_OK;
}

int ngsq_split_arrays(ngsq_engine* e, uint32_t ref, struct ngsq_split_arrays* out) {
  if (!e || !out) return NGSQ_E_ARG;
  if (!is_split(e, ref)) return fail(e, NGSQ_E_ARG, "ngsq_split_arrays: reference %u was not declared with ngsq_split_reference", ref);
  memset(out, 0, sizeof *out);
  if (e->cov_enabled[ref]) {
    out->diff = e->d_diff + e->diff_base[ref];
    out->n_diff = (uint64_t)e->ref_len[ref] + 2;
    out->tile_sums = e->d_tile_sum + e->tile_off[ref];
    out->n_tiles = cov_tiles(e, ref);
    out->touched = e->d_res + e->cov_slot[ref] + COV_TOUCHED;
  }
  if (edits_loaded(e) && e->ed_pos_total) {
    const EditsContig& ec = e->ed_contigs[ref];
    out->edit_refs = e->d_ed_refs + ec.pos_off;
    out->edit_alts = e->d_ed_alts + ec.pos_off;
    out->n_positions = (uint64_t)ec.hdr_len + 1;
  }
  return NGSQ_OK;
}

int ngsq_resolve_split(ngsq_engine* e, int is_root) {
  if (!e || !e->finished) return fail(e, NGSQ_E_ARG, "ngsq_resolve_split before finish");
  if (e->split_merged) return fail(e, NGSQ_E_ARG, "ngsq_resolve_split: the split references of this run are merged already");
  CU(cudaSetDevice(e->device));
  cudaStream_t s = e->s_comp;
  int rc = merge_split_local(e, is_root != 0, s);
  if (rc) return rc;
  if (edits_loaded(e) && e->h_ed_res.size() == E_WORDS) CU(cudaMemcpyAsync(e->h_ed_res.data(), e->d_ed_res, E_WORDS * 8, cudaMemcpyDeviceToHost, s));
  rc = ngsq_refresh_results(e);  // synchronises s
  if (rc) return rc;
  e->split_merged = true;
  e->stats.other_launches = e->other_launches;
  return NGSQ_OK;
}

void* ngsq_host_alloc(size_t nbytes) {
  void* p = nullptr;
  if (cudaHostAlloc(&p, nbytes ? nbytes : 1, cudaHostAllocDefault) != cudaSuccess) return nullptr;
  return p;
}

void ngsq_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

int ngsq_host_register(void* p, size_t nbytes) {
  return cudaHostRegister(p, nbytes, cudaHostRegisterDefault | cudaHostRegisterReadOnly) == cudaSuccess ||
                 cudaHostRegister(p, nbytes, cudaHostRegisterDefault) == cudaSuccess
             ? NGSQ_OK : NGSQ_E_CUDA;
}

int ngsq_host_unregister(void* p) { return cudaHostUnregister(p) == cudaSuccess ? NGSQ_OK : NGSQ_E_CUDA; }

int ngsq_inflate_to_host(ngsq_engine* e, const uint8_t* bgzf, size_t nbytes, uint8_t* out, size_t cap, size_t* n_out) {
  if (!e || !bgzf || !out) return fail(e, NGSQ_E_ARG, "bad arguments");
  CU(cudaSetDevice(e->device));
  DevInflated D;
  int rc = inflate_frame(e, bgzf, nbytes, 0, D);
  if (rc) return rc;
  if (n_out) *n_out = (size_t)D.total;
  if (D.total > cap) return fail(e, NGSQ_E_ARG, "output buffer too small (%llu needed)", (unsigned long long)D.total);
  if ((rc = inflate_run(e, bgzf, D))) return rc;
  if (D.total) {
    CU(cudaMemcpyAsync(out, D.out, D.total, cudaMemcpyDeviceToHost, e->s_copy));
    CU(cudaStreamSynchronize(e->s_copy));
  }
  return NGSQ_OK;
}

int ngsq_find_record(ngsq_engine* e, const uint8_t* bgzf, size_t nbytes, uint64_t file_off, uint64_t* voffset, int32_t* ref_id) {
  if (!e || !bgzf || !voffset) return fail(e, NGSQ_E_ARG, "bad arguments");
  if (!e->d_ref_len) return fail(e, NGSQ_E_ARG, "ngsq_find_record needs ngsq_set_references first (the record test needs n_ref)");
  *voffset = 0;
  if (ref_id) *ref_id = -1;
  CU(cudaSetDevice(e->device));
  DevInflated D;
  int rc = inflate_frame(e, bgzf, nbytes, file_off, D);
  if (rc) return rc;
  if (D.used != nbytes)
    return fail(e, NGSQ_E_TRUNCATED, "ngsq_find_record: the bytes at file offset %llu end inside a BGZF block", (unsigned long long)file_off);
  if ((rc = inflate_run(e, bgzf, D))) return rc;
  if (D.total < 36) return NGSQ_OK;
  cudaStream_t s = e->s_copy;
  // an 8-byte word in the spare bytes behind the decoder's queue word
  unsigned long long* d_best = reinterpret_cast<unsigned long long*>(((uintptr_t)(D.status + D.hb.size() + 1) + 7) & ~(uintptr_t)7);
  CU(cudaMemsetAsync(d_best, 0xFF, 8, s));
  const uint32_t grid = (uint32_t)std::min<uint64_t>((D.total + 255) / 256, (uint64_t)e->n_sm * 16);
  find_record_kernel<<<grid, 256, 0, s>>>(D.out, D.total, (int32_t)e->n_ref, d_best);
  CU(cudaGetLastError());
  unsigned long long best = 0;
  CU(cudaMemcpyAsync(&best, d_best, 8, cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  if (best == ~0ull) return NGSQ_OK;
  int32_t ref = -1;
  CU(cudaMemcpy(&ref, D.out + best + 4, 4, cudaMemcpyDeviceToHost));
  // the block that holds inflated offset `best` (empty blocks are not in the table)
  size_t k = 0;
  while (k + 1 < D.hb.size() && D.hb[k + 1].out_off <= best) ++k;
  *voffset = (D.hb[k].coff << 16) | (best - D.hb[k].out_off);
  if (ref_id) *ref_id = ref;
  return NGSQ_OK;
}

namespace {
// ngsq_join_bai (csi = false) and ngsq_join_csi
int join_index(ngsq_engine* const* parts, uint32_t n, uint8_t* out, size_t cap, size_t* n_out, bool csi) {
  const char* fn = csi ? "ngsq_join_csi" : "ngsq_join_bai";
  if (!parts || !n) return fail(nullptr, NGSQ_E_ARG, "%s: no parts", fn);
  ngsq_engine* e = parts[0];  // carries the message
  for (uint32_t k = 0; k < n; ++k) {
    const ngsq_engine* p = parts[k];
    if (!p) return fail(e, NGSQ_E_ARG, "%s: part %u is NULL", fn, k);
    if (!(p->cfg.flags & NGSQ_F_INDEX_PART)) return fail(e, NGSQ_E_ARG, "%s: part %u was created without NGSQ_F_INDEX_PART", fn, k);
    if (!p->finished || !p->ix_part_ok) return fail(e, NGSQ_E_ARG, "%s: part %u has no index (it did not finish without error)", fn, k);
    if (p->ref_len != parts[0]->ref_len) return fail(e, NGSQ_E_ARG, "%s: part %u has other references than part 0", fn, k);
    if (ix_csi(p) != csi)
      return fail(e, NGSQ_E_ARG, "%s: part %u builds a %s (join it with %s)", fn, k, csi ? "BAI" : "CSI", csi ? "ngsq_join_bai" : "ngsq_join_csi");
    if (csi && (p->ix_min_shift != parts[0]->ix_min_shift || p->ix_depth != parts[0]->ix_depth))
      return fail(e, NGSQ_E_ARG, "%s: part %u has min_shift %u and depth %u, part 0 has %u and %u: the parts must share one binning", fn, k,
                  p->ix_min_shift, p->ix_depth, parts[0]->ix_min_shift, parts[0]->ix_depth);
    if (k + 1 < n && p->end_voff != parts[k + 1]->first_voff)
      return fail(e, NGSQ_E_ARG, "%s: part %u ends at virtual offset %llu, part %u starts at %llu: the parts must be contiguous, in file order", fn, k,
                  (unsigned long long)p->end_voff, k + 1, (unsigned long long)parts[k + 1]->first_voff);
  }
  if (parts[n - 1]->end_voff) return fail(e, NGSQ_E_ARG, "%s: the last part must run to the end of the data (end offset 0)", fn);
  // the order across every cut: a part's first placed record against the last record before the part that constrains the
  // order (an unplaced one: ~0); every other record was checked inside its part
  uint64_t unsorted = ~0ull, last = 0;
  for (uint32_t k = 0; k < n; ++k) {
    const IxHost& H = parts[k]->ix;
    unsorted = std::min<uint64_t>(unsorted, H.S.unsorted_voff);
    if (H.S.first_voff != ~0ull && H.S.first_key < last) unsorted = std::min<uint64_t>(unsorted, H.S.first_voff);
    if (H.last_order_key) last = H.last_order_key;
  }
  if (unsorted != ~0ull) return fail_unsorted(e, unsorted);
  const ngsq_engine* p0 = parts[0];
  IxHost U;
  U.win.assign(p0->ix_win_total, ~0ull);
  U.counts.assign((size_t)p0->n_ref * 2, 0);
  U.maxw.assign(p0->n_ref, 0);
  for (uint32_t k = 0; k < n; ++k) {
    const IxHost& H = parts[k]->ix;
    U.runs.insert(U.runs.end(), H.runs.begin(), H.runs.end());
    U.ovf.insert(U.ovf.end(), H.ovf.begin(), H.ovf.end());
    for (size_t w = 0; w < U.win.size(); ++w) U.win[w] = std::min(U.win[w], H.win[w]);
    for (size_t c = 0; c < U.counts.size(); ++c) U.counts[c] += H.counts[c];
    for (size_t c = 0; c < U.maxw.size(); ++c) U.maxw[c] = std::max(U.maxw[c], H.maxw[c]);
    U.S.n_no_coor += H.S.n_no_coor;
  }
  U.data_end = parts[n - 1]->ix.data_end;
  std::vector<uint8_t> b;
  assemble_index(p0, U, b);
  if (n_out) *n_out = b.size();
  if (!out && !cap) return NGSQ_OK;
  if (!out || cap < b.size()) return fail(e, NGSQ_E_ARG, "%s: buffer holds %zu bytes, %zu needed", fn, cap, b.size());
  memcpy(out, b.data(), b.size());
  return NGSQ_OK;
}
}  // namespace

int ngsq_join_bai(ngsq_engine* const* parts, uint32_t n, uint8_t* out, size_t cap, size_t* n_out) { return join_index(parts, n, out, cap, n_out, false); }
int ngsq_join_csi(ngsq_engine* const* parts, uint32_t n, uint8_t* out, size_t cap, size_t* n_out) { return join_index(parts, n, out, cap, n_out, true); }

}  // extern "C"
