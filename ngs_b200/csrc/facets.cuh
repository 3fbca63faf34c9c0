// K4-K8 — one fused pass over the inflated records: General, Template Length, GC Content,
// Quality Score and the Coverage difference-array scatter.  Restates, per record, the
// process() bodies of the reference facets:
//   general.rs:31-124, template_length.rs:79-87, gc_content.rs:38-100,
//   quality_scores.rs:37-49, coverage.rs:148-180 (+ the query filter of command.rs:369-377).
//
// Two phases per 32 records (see facets_kernel): header-derived facets with one record per lane,
// per-base facets with one record per warp step.  Flag-derived counters: lane k owns counter k
// and adds the popcount of a ballot of bit k: no atomics for General / record tallies.  The tlen, gc
// and CIGAR-kind histograms are privatised in shared memory per CTA and flushed once with 64-bit
// global reductions; quality-by-position lives in one private table of 8-bit counters per WARP
// (plain load/add/store, flushed every 224 records).  Quality positions beyond the shared-memory
// table (long reads) go straight to the L2-resident global table.  Coverage is two signed global reductions per record into the
// contig's int32 difference array (coverage is span-based: SURVEY F6).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "recscan.cuh"

namespace ngsq {

// ---- layout of the packed u64 result buffer (also the NCCL reduce payload) ----
constexpr uint32_t R_GENERAL = 0;       // 16
constexpr uint32_t R_CIGAR = 16;        // 2 x 9
constexpr uint32_t R_TLEN_HIST = 34;    // 1025
constexpr uint32_t R_TLEN_PROCESSED = 1059;
constexpr uint32_t R_TLEN_IGNORED = 1060;
constexpr uint32_t R_GC_HIST = 1061;    // 101
constexpr uint32_t R_GC_NUC = 1162;     // gc, at, other
constexpr uint32_t R_GC_REC = 1165;     // processed, ignored_flags, ignored_too_short
constexpr uint32_t R_NONSENSICAL = 1168;
constexpr uint32_t R_ERR_QUAL = 1169;
constexpr uint32_t R_ERR_RECORD = 1170;
constexpr uint32_t R_RECORDS = 1171;
constexpr uint32_t R_QUAL_POSITIONS = 1172;  // max over records with qualities (reduced with max semantics on host)
// ngsq_reduce: rank r parks its own quality length and layout word here before the all-reduce (every other rank holds 0
// there), so ONE sum collective also tells every rank the max over ranks and whether the layouts agree
constexpr uint32_t kMaxRanks = 16;
constexpr uint32_t R_RANK_QPOS = 1176;                 // [kMaxRanks]
constexpr uint32_t R_RANK_LAYOUT = R_RANK_QPOS + kMaxRanks;  // [kMaxRanks]
constexpr uint32_t R_FIXED_WORDS = 1216;
constexpr uint32_t kReduceQualRows = 1024;  // quality rows that ride in the first collective (longer reads: one more call)
// per contig slot: [0] touched, [1] pileup_too_large, [2..2051) depth histogram, [2051..) bin sums
constexpr uint32_t COV_TOUCHED = 0, COV_TOO_LARGE = 1, COV_HIST = 2, COV_BINS = 2051;

constexpr int kFacetThreads = 224;  // 7 warps, each with a private 15 KB quality table: two CTAs per SM
constexpr uint32_t kTlenPad = 1028, kGcPad = 104, kCigWords = 18 * 32;

// A read longer than the shared-memory quality tables.  The facet kernel tallies its first qpos_smem positions and lists it
// here; qual_tiles_kernel tallies the rest and decides whether its qualities are present / in range.
struct LongRead {
  uint64_t qoff;   // slot offset of its quality string
  uint32_t ls;     // l_seq
  uint32_t flags;  // 1: some byte != 0xFF (qualities present), 2: some byte > 93
};

struct FacetParams {
  const uint8_t* d;          // base of the wave's slot
  const uint64_t* rec;       // record table of the wave: slot offset | (block + 1) << 40 (recscan.cuh)
  const RunState* st;        // wave_rec, rec_base, carry_voff, fatal
  RunState* st_w;            // the same state, for the kernel's own flags (qual_overflow)
  const BlockDesc* blocks;   // the wave's blocks (file offsets for virtual offsets)
  uint32_t headroom;
  uint32_t cov_scatter;      // 1: this kernel scatters coverage (0 with `-n`: cov_n.cuh applies the second pass's counter)
  uint64_t out0;             // offset of the wave's first block in the whole inflated stream
  uint64_t max_records;      // 0 = all
  uint64_t gc_seed;
  int32_t n_ref;
  uint32_t flags;
  const uint32_t* ref_len;
  const uint8_t* cov_enabled;
  const uint64_t* diff_base; // element offset of each contig's difference array
  int32_t* diff;
  const uint32_t* tile_off;  // index of each contig's first 4096-position tile in tile_sum
  int32_t* tile_sum;         // sum of the difference array over every tile, kept as the scatter goes (coverage.cuh)
  const uint32_t* cov_slot;  // word offset of each contig's slot in res
  uint64_t* res;
  uint64_t* qual;            // res + quality offset
  uint32_t qpos_smem;        // positions privatised in shared memory
  uint32_t qpos_cap;         // positions the global table can hold
  LongRead* long_list;       // the wave's reads with l_seq > qpos_smem (count: st_w->wave_long)
  uint32_t long_cap;
};

__device__ __forceinline__ uint64_t splitmix64_dev(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}

// Work split (ncu, profiles/: the warp-per-record form spent ~300 warp instructions per record, most
// of them on header fields with one useful lane):
//   phase A  lane <-> record: 32 records per warp step.  Header fields, validation, CIGAR (short
//            CIGARs per lane; long ones — long reads — cooperatively), coverage scatter, General
//            flag bits, template length, GC eligibility + window offset.
//   phase B  warp <-> record, 32 times: the per-base work (GC window, quality-by-position), all
//            lanes on consecutive bytes of one record.
// General / record counters are summed with one ballot + popcount per counter per 32 records.
// Quality-by-position in shared memory.  Shared-memory ATOMICS run at about one lane per clock per
// SM (ncu, profiles/: the CTA-shared u32 table made this kernel atomics-bound, 150 per record), so
// every WARP owns a private table of 8-bit counters and updates it with plain load/add/store: the
// lanes of a warp hold different positions of one record (distinct bytes), and no other warp
// touches the table.  A counter grows by at most one per record, so the warp adds its table into
// the global u64 table every kQualFlushRecords (< 256) records.  Row stride 100 bytes = 25 words
// (odd): lanes on consecutive positions with equal scores fall into different banks.
constexpr uint32_t kQualRowBytes = 100;
constexpr uint32_t kQualFlushSteps = 7;  // x 32 records per warp step = 224 < 256
__host__ __device__ inline uint32_t qual_table_bytes(uint32_t qpos_smem) { return (qpos_smem * kQualRowBytes + 15u) & ~15u; }

constexpr uint32_t kShortCigar = 8;    // CIGARs up to this many ops are tallied by the record's own lane

// adds a warp's private 8-bit table into the global table and clears it: one row (position) per
// lane, so that all lanes stay busy (a row holds a handful of non-zero counters)
__device__ __forceinline__ void flush_qual_table(uint32_t* tab_words, uint32_t n_rows, unsigned long long* gqual, uint32_t lane) {
  for (uint32_t row = lane; row < n_rows; row += 32) {
    uint32_t* rw = tab_words + row * (kQualRowBytes / 4);
    for (uint32_t wi = 0; wi < 94 / 4 + 1; ++wi) {
      const uint32_t v = rw[wi];
      if (v) {
        rw[wi] = 0;
#pragma unroll
        for (uint32_t k = 0; k < 4; ++k) {
          const uint32_t c = (v >> (8 * k)) & 255u;
          if (c) atomicAdd(&gqual[(uint64_t)row * 94 + wi * 4 + k], (unsigned long long)c);
        }
      }
    }
  }
  __syncwarp();
}

constexpr uint32_t kQualPre = 5;  // quality positions per lane loaded one record ahead (covers reads up to 160 bases)
// positions privatised in shared memory (per warp: 152 x 100 B; two 7-warp CTAs per SM); the rest goes to the global table.
// Fixed: the engine streams the file and cannot know the longest read when it launches the first wave.
constexpr uint32_t kQualSmemPositions = 152;

// loads of one record that phase B needs: the quality bytes at positions lane + 32k, k < kQualPre.  Unconditional
// (bytes behind a short string belong to the next record or to the slot's slack; they are masked when they are
// tallied): one base address, five immediate offsets, no predicates.  Nothing here may consume a loaded value (no
// selects, no shifts): the loads must stay in flight while the previous record is tallied.
__device__ __forceinline__ void facet_prefetch(const uint8_t* sq, uint32_t ls, uint32_t lane, uint32_t (&qb)[kQualPre]) {
  const uint8_t* qlane = sq + (ls + 1) / 2 + lane;
#pragma unroll
  for (uint32_t k = 0; k < kQualPre; ++k) qb[k] = __ldg(qlane + 32 * k);
}

// G/C and A/T bases among the 100 bases that start at base `gj` of a 4-bit packed sequence (gc_content.rs:76-100), by the
// record's own lane: 13 unaligned words over the window's whole bytes (49 or 50), the two odd nibbles at its ends.
// A, C, G, T are the one-hot codes 1, 2, 4, 8: per nibble, C|G <=> exactly one of bits 1, 2 and neither of bits 0, 3;
// A|T <=> exactly one of bits 0, 3 and neither of bits 1, 2 (eight nibbles of a word at once).
__device__ __forceinline__ void gc_window_counts(const uint8_t* seq, uint32_t gj, uint32_t* gc_out, uint32_t* at_out) {
  const uint32_t odd = gj & 1u;
  const uint8_t* fp = seq + ((gj + 1) >> 1);  // first whole byte of the window
  const uint32_t* w = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(fp) & ~uintptr_t(3));
  const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(fp) & 3) * 8;
  uint32_t gc = 0, at = 0, g_acc = 0, a_acc = 0;
  uint32_t prev = __ldg(w);
#pragma unroll
  for (int i = 0; i < 13; ++i) {
    const uint32_t nxt = __ldg(w + i + 1);
    uint32_t u = __funnelshift_r(prev, nxt, sh);
    prev = nxt;
    if (i == 12) u &= odd ? 0xFFu : 0xFFFFu;  // bytes 48 (and 49): 49 whole bytes when the window starts on a low nibble
    const uint32_t b1 = u >> 1, b2 = u >> 2, b3 = u >> 3;
    g_acc |= ((b1 ^ b2) & ~(u | b3) & 0x11111111u) << (i & 3);
    a_acc |= ((u ^ b3) & ~(b1 | b2) & 0x11111111u) << (i & 3);
    if ((i & 3) == 3 || i == 12) {
      gc += __popc(g_acc);
      at += __popc(a_acc);
      g_acc = a_acc = 0;
    }
  }
  if (odd) {  // first base: low nibble of the byte before; last base: high nibble of the byte behind the whole bytes
    const uint32_t n1 = __ldg(seq + (gj >> 1)) & 15u, n2 = (uint32_t)__ldg(seq + ((gj + 99) >> 1)) >> 4;
    gc += (n1 == 2u || n1 == 4u) + (n2 == 2u || n2 == 4u);
    at += (n1 == 1u || n1 == 8u) + (n2 == 1u || n2 == 8u);
  }
  *gc_out = gc;
  *at_out = at;
}

// ---- per-record rules, shared by facets_kernel and the per-read-group pass (read_groups.cuh) ----
// The fixed 36 header bytes of the record at p (its block_size word) at any alignment: ten aligned words, nine funnel shifts.
// Returns false when the fields overrun block_size or a reference id is out of range (the run fails with NGSQ_E_BAD_RECORD).
struct RecHeader {
  uint32_t bs, lseq, f, ncig, lname, mapq;
  int32_t ref, pos, nref, tlen;
};
__device__ __forceinline__ bool load_record_header(const uint8_t* p, int32_t n_ref, RecHeader& h) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(p) & ~uintptr_t(3));
  const uint32_t sh = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 3) * 8;
  const uint32_t a0 = w[0], a1 = w[1], a2 = w[2], a3 = w[3], a4 = w[4], a5 = w[5], a6 = w[6], a7 = w[7], a8 = w[8], a9 = w[9];
  h.bs = __funnelshift_r(a0, a1, sh);
  h.ref = (int32_t)__funnelshift_r(a1, a2, sh);
  h.pos = (int32_t)__funnelshift_r(a2, a3, sh);
  const uint32_t w3 = __funnelshift_r(a3, a4, sh);
  const uint32_t w4 = __funnelshift_r(a4, a5, sh);
  h.lseq = __funnelshift_r(a5, a6, sh);
  h.nref = (int32_t)__funnelshift_r(a6, a7, sh);
  h.tlen = (int32_t)__funnelshift_r(a8, a9, sh);
  h.lname = w3 & 255; h.mapq = (w3 >> 8) & 255; h.ncig = w4 & 0xFFFF; h.f = w4 >> 16;
  const uint64_t need = 32ull + h.lname + 4ull * h.ncig + (h.lseq + 1ull) / 2 + h.lseq;
  return !(need > h.bs || h.ref < -1 || h.ref >= n_ref || h.nref < -1 || h.nref >= n_ref);
}

// General counters (general.rs:31-101): bit k set <=> counter k of ngsq_get_general counts the record.  A mapped pair
// without reference ids sets err_rec (the reference panics there, general.rs:81-83).
__device__ __forceinline__ uint32_t general_bits(uint32_t f, int32_t ref, int32_t nref, uint32_t mapq, uint32_t& err_rec) {
  uint32_t bits = 1u;
  if (f & 0x4) bits |= 1u << 1;
  if (f & 0x400) bits |= 1u << 2;
  if (f & 0x100) bits |= 1u << 4;
  else if (f & 0x800) bits |= 1u << 5;
  else {
    bits |= 1u << 3;
    if (!(f & 0x4)) bits |= 1u << 6;
    if (f & 0x400) bits |= 1u << 7;
    if (f & 0x1) {
      bits |= 1u << 8;
      if (f & 0x40) bits |= 1u << 9;
      if (f & 0x80) bits |= 1u << 10;
      if (!(f & 0x4)) {
        if (f & 0x2) bits |= 1u << 11;
        if (f & 0x8) bits |= 1u << 12;
        else {
          bits |= 1u << 13;
          if (ref < 0 || nref < 0) err_rec = 1;  // the reference panics here (general.rs:81-83)
          else if (ref != nref) {
            bits |= 1u << 14;
            if (mapq >= 5) bits |= 1u << 15;     // missing (255) counts (general.rs:88-95)
          }
        }
      }
    }
  }
  return bits;
}

// Template length (template_length.rs:79-87, `tlen as usize`, bins 0..=1024): bit 16 processed (bin = tlen), bit 17 ignored
__device__ __forceinline__ uint32_t tlen_bits(int32_t tlen) { return (tlen >= 0 && tlen <= 1024) ? 1u << 16 : 1u << 17; }

// GC content eligibility (gc_content.rs:38-75): bit 18 processed, 19 ignored (flags), 20 ignored (too short)
__device__ __forceinline__ uint32_t gc_bits(uint32_t f, uint32_t lseq) {
  if (f & (0x400 | 0x100)) return 1u << 19;
  if (lseq < 100) return 1u << 20;
  return 1u << 18;
}

// Window offset of a GC-processed read with l_seq > 100 (gc_content.rs:69-74, see ngsq_get_gc): keyed by the record's BGZF
// virtual offset, i.e. its block's file offset and its offset in that block (the record carried into the wave: carry_voff)
__device__ __forceinline__ uint32_t gc_window_offset(uint64_t rv, const BlockDesc* blocks, uint64_t carry_voff, uint32_t headroom,
                                                     uint64_t out0, uint64_t gc_seed, uint32_t lseq) {
  const uint32_t t = (uint32_t)(rv >> 40);
  uint64_t voff = carry_voff;
  if (t) { const BlockDesc& bd = blocks[t - 1]; voff = (bd.coff << 16) | ((rv & kRecOffMask) - headroom - (bd.out_off - out0)); }
  return (uint32_t)(((splitmix64_dev(gc_seed ^ voff) >> 32) * (uint64_t)(lseq - 100)) >> 32);
}

__global__ void __launch_bounds__(kFacetThreads) facets_kernel(FacetParams P) {
  extern __shared__ uint32_t sm[];
  const uint32_t warps_in_cta = blockDim.x >> 5;
  const uint32_t qtab_words = qual_table_bytes(P.qpos_smem) / 4;
  uint32_t* s_tlen = sm + qtab_words * warps_in_cta;
  uint32_t* s_gc = s_tlen + kTlenPad;
  uint32_t* s_cig = s_gc + kGcPad;
  const uint32_t n_sm = qtab_words * warps_in_cta + kTlenPad + kGcPad + kCigWords;
  uint32_t* my_qwords = sm + qtab_words * (threadIdx.x >> 5);          // this warp's private table
  uint8_t* my_qtab = reinterpret_cast<uint8_t*>(my_qwords);
  uint8_t* my_qrow = my_qtab + (threadIdx.x & 31) * kQualRowBytes;  // row of position `lane`; position lane + 32k is 32k rows further
  uint32_t steps_since_flush = 0;
  for (uint32_t i = threadIdx.x; i < n_sm; i += blockDim.x) sm[i] = 0;
  __syncthreads();

  const uint32_t lane = threadIdx.x & 31;
  const uint32_t warps_per_cta = blockDim.x >> 5;
  const uint64_t n_warps = (uint64_t)gridDim.x * warps_per_cta;
  const bool do_rec = P.flags & 1u;
  uint32_t acc = 0;                        // lane k owns counter k (bit k of every record's `bits`)
  uint32_t sum_gc = 0, sum_at = 0, sum_oth = 0;  // per lane (the record's own lane counts its GC window)
  uint32_t err_qual = 0, err_rec = 0, max_qpos = 0, qual_over = 0;
  const uint64_t n_rec = P.st->fatal ? 0 : P.st->wave_rec, rec_base = P.st->rec_base;
  const bool do_cov = (P.flags & 2u) && P.cov_scatter;

  for (uint64_t r0 = ((uint64_t)blockIdx.x * warps_per_cta + (threadIdx.x >> 5)) * 32; r0 < n_rec; r0 += n_warps * 32) {
    // ================= phase A: one record per lane =================
    const uint64_t r = r0 + lane;
    bool valid = r < n_rec;
    const uint8_t* p = P.d;
    uint32_t lseq = 0, f = 0, ncig = 0, lname = 0, mapq = 0;
    uint64_t rv = 0;
    int32_t ref = -1, pos = -1, nref = -1, tlen = 0;
    if (valid) {
      rv = P.rec[r];
      p = P.d + (rv & kRecOffMask);
      RecHeader h;
      if (!load_record_header(p, P.n_ref, h)) { err_rec = 1; valid = false; }
      ref = h.ref; pos = h.pos; lseq = h.lseq; nref = h.nref; tlen = h.tlen;
      lname = h.lname; mapq = h.mapq; ncig = h.ncig; f = h.f;
    }
    const uint8_t* cig = p + 36 + lname;
    const uint8_t* seq = cig + 4 * (size_t)ncig;
    const uint8_t* qual = seq + (lseq + 1) / 2;
    const bool in_n = P.max_records == 0 || rec_base + r < P.max_records;
    const bool rec_on = valid && do_rec && in_n;

    // ---- long reads: listed for qual_tiles_kernel (positions >= qpos_smem of their quality strings)
    {
      const bool is_long = rec_on && lseq > P.qpos_smem;
      const uint32_t m = __ballot_sync(0xFFFFFFFFu, is_long);
      if (m) {  // warp-uniform; never taken on short-read data
        const int leader = __ffs(m) - 1;
        uint32_t base = 0;
        if ((int)lane == leader) base = atomicAdd(&P.st_w->wave_long, (uint32_t)__popc(m));
        base = __shfl_sync(0xFFFFFFFFu, base, leader);
        if (is_long) {
          const uint32_t idx = base + __popc(m & ((1u << lane) - 1));
          if (idx < P.long_cap) P.long_list[idx] = LongRead{(uint64_t)(qual - P.d), lseq, 0u};
          else atomicOr(&P.st_w->fatal, kFatalRecTable);  // sized by bytes / (smallest long record): cannot happen
          if (lseq > P.qpos_cap) qual_over = lseq > qual_over ? lseq : qual_over;  // the run fails with a request for a longer table
        }
      }
    }

    // ---- CIGAR: kind tallies (general.rs:103-121) and reference span (utils/cigar.rs:6-11)
    uint32_t span = 0;
    const uint32_t which = (f & 0x40) ? 0 : 9;
    if (valid && ncig <= kShortCigar) {
      for (uint32_t i = 0; i < ncig; ++i) {
        const uint32_t op = ld_u32_unaligned(cig + 4 * i);
        const uint32_t k = op & 15;
        if (k > 8) { err_rec = 1; continue; }
        if ((0x18D >> k) & 1) span += op >> 4;  // M D N = X
        if (rec_on) atomicAdd(&s_cig[(which + k) * 32 + lane], 1u);
      }
    }
    // long CIGARs (long reads): the whole warp strides over one record's ops
    for (uint32_t todo = __ballot_sync(0xFFFFFFFFu, valid && ncig > kShortCigar); todo; todo &= todo - 1) {
      const int j = __ffs(todo) - 1;
      const uint8_t* cj = reinterpret_cast<const uint8_t*>(__shfl_sync(0xFFFFFFFFu, (unsigned long long)cig, j));
      const uint32_t nj = __shfl_sync(0xFFFFFFFFu, ncig, j);
      const uint32_t wj = __shfl_sync(0xFFFFFFFFu, which, j);
      const bool onj = __shfl_sync(0xFFFFFFFFu, (int)rec_on, j);
      uint32_t sp = 0, bad = 0;
      for (uint32_t i = lane; i < nj; i += 32) {
        const uint32_t op = ld_u32_unaligned(cj + 4 * i);
        const uint32_t k = op & 15;
        if (k > 8) { bad = 1; continue; }
        if ((0x18D >> k) & 1) sp += op >> 4;
        if (onj) atomicAdd(&s_cig[(wj + k) * 32 + lane], 1u);
      }
      sp = __reduce_add_sync(0xFFFFFFFFu, sp);
      if (__any_sync(0xFFFFFFFFu, bad)) err_rec = 1;
      if ((int)lane == j) span = sp;
    }

    // ---- Coverage scatter (coverage.rs:148-180 behind the query filter, SURVEY App. D.6)
    {
      uint32_t t_up = 0xFFFFFFFFu, t_dn = 0xFFFFFFFFu;  // tiles whose sums take this record's +1 / -1
      if (do_cov && valid && ref >= 0 && pos >= 0 && P.cov_enabled[ref]) {
        const int64_t L = P.ref_len[ref];
        const int64_t start = (int64_t)pos + 1, end = start + (int64_t)span - 1;
        if (start <= L && end >= 1) {
          P.res[P.cov_slot[ref] + COV_TOUCHED] = 1;
          if (span) {
            int32_t* df = P.diff + P.diff_base[ref];
            atomicAdd(df + start, 1);
            const int64_t e = end < L ? end : L;
            atomicAdd(df + e + 1, -1);
            if (end > L) atomicAdd((unsigned long long*)&P.res[R_NONSENSICAL], (unsigned long long)(end - L));
            t_up = P.tile_off[ref] + (uint32_t)(start >> 12);
            if (e + 1 <= L) t_dn = P.tile_off[ref] + (uint32_t)((e + 1) >> 12);  // position L + 1 lies outside the resolved range
          }
        }
      }
      // a sorted file sends a warp's 32 records to one or two tiles: one reduction per distinct tile, not per record
      if (do_cov) {
        const uint32_t m_up = __ballot_sync(0xFFFFFFFFu, t_up != 0xFFFFFFFFu), m_dn = __ballot_sync(0xFFFFFFFFu, t_dn != 0xFFFFFFFFu);
        if (t_up != 0xFFFFFFFFu) {
          const uint32_t peers = __match_any_sync(m_up, t_up);
          if ((int)lane == __ffs(peers) - 1) atomicAdd(P.tile_sum + t_up, (int)__popc(peers));
        }
        if (t_dn != 0xFFFFFFFFu) {
          const uint32_t peers = __match_any_sync(m_dn, t_dn);
          if ((int)lane == __ffs(peers) - 1) atomicAdd(P.tile_sum + t_dn, -(int)__popc(peers));
        }
      }
    }
    if (!do_rec) continue;

    // ---- General counters (general.rs:31-101): bit k of `bits` increments counter k
    uint32_t bits = 0;
    bool gc_on = false;
    uint32_t gc_off = 0;
    if (rec_on) {
      bits = general_bits(f, ref, nref, mapq, err_rec);
      bits |= tlen_bits(tlen);
      if (bits & (1u << 16)) atomicAdd(&s_tlen[tlen], 1u);
      bits |= gc_bits(f, lseq);
      if (bits & (1u << 18)) {
        gc_on = true;
        if (lseq > 100) gc_off = gc_window_offset(rv, P.blocks, P.st->carry_voff, P.headroom, P.out0, P.gc_seed, lseq);
      }
    }
#pragma unroll
    for (int k = 0; k < 21; ++k) {
      const uint32_t m = __ballot_sync(0xFFFFFFFFu, (bits >> k) & 1u);
      if ((int)lane == k) acc += __popc(m);
    }
    // ---- GC window (gc_content.rs:76-100): the record's own lane counts its 100 bases
    if (gc_on) {
      uint32_t gc, at;
      gc_window_counts(seq, gc_off, &gc, &at);
      sum_gc += gc; sum_at += at; sum_oth += 100 - gc - at;
      atomicAdd(&s_gc[gc], 1u);  // round(gc / 100 * 100) == gc
    }

    // ================= phase B: one record per warp step =================
    // Quality by position.  Software-pipelined two records deep: the first 160 quality positions of the NEXT TWO records
    // are loaded before the current two are tallied (ncu: with one record in flight per warp the kernel sat on the long
    // scoreboard at the first use of the prefetched bytes — 14 warps per SM cannot hide an HBM round trip otherwise).
    uint32_t todo = __ballot_sync(0xFFFFFFFFu, rec_on && lseq != 0);
    const uint32_t n_pre = P.qpos_smem < 32 * kQualPre ? P.qpos_smem : 32 * kQualPre;  // positions the prefetch covers
    // takes the next record off `todo` (warp-uniform) and issues its loads
    auto fetch = [&](const uint8_t*& sq, uint32_t& ls, uint32_t (&qb)[kQualPre]) -> bool {
      const bool on = todo != 0;
      const int j = on ? __ffs(todo) - 1 : 0;
      todo &= todo - 1;
      sq = reinterpret_cast<const uint8_t*>(__shfl_sync(0xFFFFFFFFu, (unsigned long long)seq, j));
      ls = __shfl_sync(0xFFFFFFFFu, lseq, j);
      if (on) facet_prefetch(sq, ls, lane, qb);
      return on;
    };
    // Quality scores of one record (quality_scores.rs:37-49; presence rule SURVEY App. D.5): one pass.
    // Qualities are present unless every byte is 0xFF; a present string must be <= 93 throughout,
    // so increments for bytes <= 93 are exact whenever the run does not fail.
    // per lane: smallest byte seen (0x100 = none) and largest real byte; "present" <=> some byte != 0xFF,
    // "too big" <=> some byte in 94..255 — two min/max per position instead of compares and branches
    auto tally = [&](const uint8_t* sq, uint32_t ls, const uint32_t (&qb)[kQualPre]) {
      const uint32_t n_s = ls < n_pre ? ls : n_pre;
      uint32_t q_min = 0x100u, q_max = 0;
#pragma unroll
      for (uint32_t k = 0; k < kQualPre; ++k) {
        const uint32_t q = lane + 32 * k < n_s ? qb[k] : 0x100u;  // beyond the string (or the shared-memory table)
        q_min = min(q_min, q);
        q_max = max(q_max, q & 0xFFu);  // the "beyond the string" marker 0x100 counts as 0 here
        if (q <= 93) {
          uint8_t* c = my_qrow + k * (32 * kQualRowBytes) + q;  // private to this warp; lanes hold distinct positions
          *c = (uint8_t)(*c + 1);
        }
      }
      bool any_real = q_min < 0xFFu, any_big = q_max > 93;
      if (ls > n_pre) {  // warp-uniform: short reads never enter
        const uint8_t* ql = sq + (ls + 1) / 2;
        const uint32_t n_t = ls < P.qpos_smem ? ls : P.qpos_smem;
        for (uint32_t i = n_pre + lane; i < n_t; i += 32) {  // shared-memory positions beyond the prefetched ones
          const uint32_t q = __ldg(ql + i);
          any_real |= q != 0xFF;
          if (q > 93) any_big = true;
          else {
            uint8_t* c = my_qtab + i * kQualRowBytes + q;
            *c = (uint8_t)(*c + 1);
          }
        }
        // positions >= qpos_smem: qual_tiles_kernel, which also gives the verdict below for such a read (ncu, configs[3]:
        // one global reduction per base ran at the L2's atomic rate, ~120 G/s whatever the operand width)
      }
      if (ls <= P.qpos_smem) {  // warp-uniform
        any_real = __any_sync(0xFFFFFFFFu, any_real);
        any_big = __any_sync(0xFFFFFFFFu, any_big);
        if (any_real) {
          if (any_big) err_qual = 1;
          max_qpos = ls > max_qpos ? ls : max_qpos;
        }
      }
    };
    const uint8_t *sq_a, *sq_b;
    uint32_t ls_a, ls_b, qb_a[kQualPre], qb_b[kQualPre];
    bool on_a = fetch(sq_a, ls_a, qb_a), on_b = fetch(sq_b, ls_b, qb_b);
    while (on_a) {
      const uint8_t *sq_c, *sq_d;
      uint32_t ls_c, ls_d, qb_c[kQualPre], qb_d[kQualPre];
      const bool on_c = fetch(sq_c, ls_c, qb_c), on_d = fetch(sq_d, ls_d, qb_d);
      tally(sq_a, ls_a, qb_a);
      if (on_b) tally(sq_b, ls_b, qb_b);
      sq_a = sq_c; ls_a = ls_c; on_a = on_c;
      sq_b = sq_d; ls_b = ls_d; on_b = on_d;
#pragma unroll
      for (uint32_t k = 0; k < kQualPre; ++k) { qb_a[k] = qb_c[k]; qb_b[k] = qb_d[k]; }
    }
    __syncwarp();
    if (++steps_since_flush == kQualFlushSteps) {
      flush_qual_table(my_qwords, P.qpos_smem, (unsigned long long*)P.qual, lane);
      steps_since_flush = 0;
    }
  }
  if (do_rec && steps_since_flush) flush_qual_table(my_qwords, P.qpos_smem, (unsigned long long*)P.qual, lane);

  // ---- flush ----
  __syncthreads();
  if (do_rec) {
    // lane-owned counters: 0..15 general, 16/17 tlen processed/ignored, 18..20 gc records
    if (acc) {
      uint32_t slot;
      if (lane < 16) slot = R_GENERAL + lane;
      else if (lane == 16) slot = R_TLEN_PROCESSED;
      else if (lane == 17) slot = R_TLEN_IGNORED;
      else slot = R_GC_REC + (lane - 18);
      if (lane < 21) atomicAdd((unsigned long long*)&P.res[slot], (unsigned long long)acc);
    }
    sum_gc = __reduce_add_sync(0xFFFFFFFFu, sum_gc);
    sum_at = __reduce_add_sync(0xFFFFFFFFu, sum_at);
    sum_oth = __reduce_add_sync(0xFFFFFFFFu, sum_oth);
    if (lane == 0) {
      if (sum_gc) atomicAdd((unsigned long long*)&P.res[R_GC_NUC + 0], (unsigned long long)sum_gc);
      if (sum_at) atomicAdd((unsigned long long*)&P.res[R_GC_NUC + 1], (unsigned long long)sum_at);
      if (sum_oth) atomicAdd((unsigned long long*)&P.res[R_GC_NUC + 2], (unsigned long long)sum_oth);
    }
    for (uint32_t i = threadIdx.x; i < 1025; i += blockDim.x)
      if (s_tlen[i]) atomicAdd((unsigned long long*)&P.res[R_TLEN_HIST + i], (unsigned long long)s_tlen[i]);
    for (uint32_t i = threadIdx.x; i < 101; i += blockDim.x)
      if (s_gc[i]) atomicAdd((unsigned long long*)&P.res[R_GC_HIST + i], (unsigned long long)s_gc[i]);
    if (threadIdx.x < 18) {
      uint32_t t = 0;
      for (uint32_t l = 0; l < 32; ++l) t += s_cig[threadIdx.x * 32 + l];
      if (t) atomicAdd((unsigned long long*)&P.res[R_CIGAR + threadIdx.x], (unsigned long long)t);
    }
    if (max_qpos) atomicMax((unsigned long long*)&P.res[R_QUAL_POSITIONS], (unsigned long long)max_qpos);
  }
  if (err_qual) P.res[R_ERR_QUAL] = 1;
  if (err_rec) P.res[R_ERR_RECORD] = 1;
  if (qual_over) atomicMax(&P.st_w->qual_overflow, qual_over);
}

// ---- quality positions beyond the shared-memory tables (long reads) ----
// Work item = (tile of kTilePos positions) x (chunk of the wave's LongRead list).  A CTA tallies an item into 32-bit
// shared-memory counters (lanes of one instruction hold distinct positions: no same-address conflicts), then adds the
// non-zero counters to the global table: one global reduction per (item, position, score) instead of one per base.
// (Measured alternative, rejected: one lane per position with plain load / add / store on a lane-owned row and all warps
// walking every read of the item — no atomics, but eight times the serial iterations per warp: configs[3]'s facet stage
// 511 ms against ~250 ms with this form.)
constexpr uint32_t kTilePos = 256;
constexpr uint32_t kTileThreads = 256;
constexpr uint32_t kTileSmem = kTilePos * 94 * 4;  // 94 KB: two CTAs per SM

struct QualTileParams {
  const uint8_t* d;      // base of the wave's slot
  LongRead* list;
  uint32_t long_cap;
  const RunState* st;    // wave_long, max_lseq, fatal
  uint64_t* qual;        // global table [qpos_cap][94]
  uint64_t* res;
  uint32_t qpos_smem, qpos_cap;
};

__global__ void __launch_bounds__(kTileThreads) qual_tiles_kernel(QualTileParams P) {
  extern __shared__ uint32_t t_cnt[];  // [kTilePos][94]
  const uint32_t n_long = P.st->wave_long < P.long_cap ? P.st->wave_long : P.long_cap;
  const uint32_t top = P.st->max_lseq < P.qpos_cap ? P.st->max_lseq : P.qpos_cap;  // longest read so far (never less than this wave's)
  if (!n_long || P.st->fatal || top <= P.qpos_smem) return;
  const uint32_t n_tiles = (top - P.qpos_smem + kTilePos - 1) / kTilePos;
  // enough chunks that every CTA finds several items (high tiles hold few reads), but at least 64 reads per item
  uint32_t n_chunks = (4 * gridDim.x + n_tiles - 1) / n_tiles;
  const uint32_t max_chunks = (n_long + 63) / 64;
  if (n_chunks > max_chunks) n_chunks = max_chunks;
  const uint32_t per = (n_long + n_chunks - 1) / n_chunks;
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (uint32_t i = threadIdx.x; i < kTilePos * 94; i += kTileThreads) t_cnt[i] = 0;
  __syncthreads();
  for (uint32_t item = blockIdx.x; item < n_tiles * n_chunks; item += gridDim.x) {
    const uint32_t tile = item / n_chunks, chunk = item - tile * n_chunks;
    const uint32_t p_lo = P.qpos_smem + tile * kTilePos;
    const uint32_t r0 = chunk * per, r1 = r0 + per < n_long ? r0 + per : n_long;
    for (uint32_t r = r0 + warp; r < r1; r += kTileThreads / 32) {
      const uint32_t ls = P.list[r].ls;
      if (ls <= p_lo) continue;  // warp-uniform
      const uint8_t* ql = P.d + P.list[r].qoff;
      uint32_t p_hi = ls < p_lo + kTilePos ? ls : p_lo + kTilePos;
      if (p_hi > P.qpos_cap) p_hi = P.qpos_cap;
      uint32_t q[kTilePos / 32];
#pragma unroll
      for (uint32_t k = 0; k < kTilePos / 32; ++k) {
        const uint32_t p = p_lo + lane + 32 * k;
        q[k] = p < p_hi ? (uint32_t)__ldg(ql + p) : 0x100u;  // 0x100: beyond the string
      }
      uint32_t q_min = 0x100u, q_max = 0;
#pragma unroll
      for (uint32_t k = 0; k < kTilePos / 32; ++k) {
        q_min = min(q_min, q[k]);
        q_max = max(q_max, q[k] & 0xFFu);
        if (q[k] <= 93) atomicAdd(&t_cnt[(lane + 32 * k) * 94 + q[k]], 1u);
      }
      if (tile == 0)  // the positions the facet kernel tallied: only their share of the verdict
        for (uint32_t p = lane; p < P.qpos_smem; p += 32) {
          const uint32_t v = __ldg(ql + p);
          q_min = min(q_min, v);
          q_max = max(q_max, v);
        }
      uint32_t f = (q_min < 0xFFu ? 1u : 0u) | (q_max > 93 ? 2u : 0u);
      f = __reduce_or_sync(0xFFFFFFFFu, f);
      if (f && lane == 0) {
        const uint32_t have = *(volatile uint32_t*)&P.list[r].flags;  // other tiles of the same read set the same bits
        if ((have | f) != have) atomicOr(&P.list[r].flags, f);
      }
    }
    __syncthreads();
    const uint32_t rows = top - p_lo < kTilePos ? top - p_lo : kTilePos;
    unsigned long long* g = (unsigned long long*)P.qual + (uint64_t)p_lo * 94;
    for (uint32_t i = threadIdx.x; i < rows * 94; i += kTileThreads) {
      const uint32_t v = t_cnt[i];
      if (v) { t_cnt[i] = 0; atomicAdd(&g[i], (unsigned long long)v); }
    }
    __syncthreads();
  }
}

// Present / in-range verdict of the wave's long reads (quality_scores.rs:37-49; SURVEY App. D.5), after every tile is in.
__global__ void __launch_bounds__(256) qual_verdict_kernel(QualTileParams P) {
  const uint32_t n_long = P.st->wave_long < P.long_cap ? P.st->wave_long : P.long_cap;
  if (!n_long || P.st->fatal) return;
  uint32_t err = 0, mx = 0;
  for (uint32_t r = blockIdx.x * blockDim.x + threadIdx.x; r < n_long; r += gridDim.x * blockDim.x) {
    const uint32_t f = P.list[r].flags;
    if (f & 1u) {
      if (f & 2u) err = 1;
      mx = P.list[r].ls > mx ? P.list[r].ls : mx;
    }
  }
  mx = __reduce_max_sync(0xFFFFFFFFu, mx);
  err = __any_sync(0xFFFFFFFFu, err);
  if ((threadIdx.x & 31) == 0) {
    if (mx) atomicMax((unsigned long long*)&P.res[R_QUAL_POSITIONS], (unsigned long long)mx);
    if (err) P.res[R_ERR_QUAL] = 1;
  }
}

}  // namespace ngsq
