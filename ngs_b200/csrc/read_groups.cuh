// NGSQ_F_READ_GROUPS — the four record facets (General, Template Length, GC Content, Quality Score) once more per read group,
// behind facets_kernel on the same wave (DESIGN.md section 5, "Read groups").  Four kernels per wave:
//   rg_tag_kernel      one lane per record: the group of its first `RG` aux field (htslib's bam_aux_get), counted per group
//   rg_scan_kernel     one CTA: bucket offsets over the n + 1 counts, each bucket padded to whole warp steps of 32 records
//   rg_scatter_kernel  one lane per record: its record-table index into its group's bucket
//   rg_facets_kernel   phase A / phase B of facets_kernel over the buckets: a warp step holds records of ONE group, so the
//                      flag counters are one ballot per counter, and the quality table and the TLEN and GC histograms
//                      per-warp 8-bit tables; all are flushed into the group's slice when the warp's group changes and
//                      every kQualFlushSteps steps.
// The per-record rules are facets.cuh's (load_record_header, general_bits, tlen_bits, gc_bits, gc_window_offset,
// gc_window_counts); the quality rule is quality_scores.rs:37-49 as facets_kernel applies it (bytes <= 93 are counted, a read
// counts towards the group's quality length when some byte is not 0xFF; a byte > 93 fails the run in facets_kernel).
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "facets.cuh"

namespace ngsq {

// ---- one group's slice of the group buffer ----
// [0, kGroupSums): the u64 counters of the packed result buffer's fixed part, at the same offsets (R_GENERAL .. R_GC_REC + 3);
// the quality lengths of all groups follow the sums of all groups, the quality tables ([rows][94] each) follow those.
constexpr uint32_t kGroupSums = R_NONSENSICAL;  // 1168
constexpr uint16_t kNoGroup = 0xFFFF;           // record outside `-n`, or invalid
constexpr uint32_t kRgEmpty = 0;                // free slot of the ID hash table
constexpr uint32_t kRgThreads = 256;
constexpr uint32_t kRgScanThreads = 1024;

__host__ __device__ inline uint32_t rg_hash(const uint8_t* s, uint32_t n) {  // FNV-1a
  uint32_t h = 2166136261u;
  for (uint32_t i = 0; i < n; ++i) h = (h ^ s[i]) * 16777619u;
  return h;
}

struct ReadGroupParams {
  const uint8_t* d;          // base of the wave's slot
  const uint64_t* rec;       // record table of the wave (recscan.cuh)
  const RunState* st;
  const BlockDesc* blocks;
  uint32_t headroom;
  uint64_t out0;
  uint64_t max_records;      // 0 = all
  uint64_t gc_seed;
  int32_t n_ref;
  uint32_t n_groups;         // declared IDs; group n_groups = ungrouped
  const uint8_t* ids;        // the IDs back to back, NUL-terminated
  const uint32_t* id_off;    // [n_groups + 1] offsets into ids
  const uint32_t* table;     // [mask + 1] open-addressing table: group + 1, or kRgEmpty
  uint32_t mask;
  uint16_t* grp;             // [record] group of the record, kNoGroup = none
  uint32_t* count;           // [n_groups + 1] records per group in this wave (zeroed again by rg_scan_kernel)
  uint32_t* cursor;          // [n_groups + 1] next free slot of each bucket
  uint32_t* order;           // record-table indices, bucket after bucket, 0xFFFFFFFF in the padding
  uint32_t* total;           // slots of all buckets (a multiple of 32)
  uint64_t* sums;            // [n_groups + 1][kGroupSums]
  uint64_t* qlen;            // [n_groups + 1] longest read with qualities
  uint64_t* qual;            // [n_groups + 1][rows][94]
  uint32_t rows;             // = the sample's quality rows (qpos_cap)
  uint64_t* res;             // the sample's result buffer: R_ERR_RECORD for a malformed aux field
};

// Group of the record at p whose aux fields are [a, end): htslib's bam_aux_get — the first field tagged RG decides; a type
// other than Z, a missing NUL or a value that matches no declared ID byte for byte gives the ungrouped group n.  A malformed
// field in front of it (unknown type, missing NUL, a field that runs past the record) sets *bad.
__device__ __forceinline__ uint32_t rg_lookup(const uint8_t* a, const uint8_t* end, const ReadGroupParams& P, bool* bad) {
  const uint32_t none = P.n_groups;
  while (a < end) {
    if (end - a < 3) { *bad = true; return none; }
    const uint8_t t0 = a[0], t1 = a[1], ty = a[2];
    a += 3;
    if (t0 == 'R' && t1 == 'G') {
      if (ty != 'Z') return none;
      uint32_t h = 2166136261u, n = 0;
      for (; a + n < end && a[n]; ++n) h = (h ^ a[n]) * 16777619u;
      if (a + n >= end) return none;  // no NUL inside the record
      for (uint32_t s = h & P.mask;; s = (s + 1) & P.mask) {
        const uint32_t v = P.table[s];
        if (v == kRgEmpty) return none;
        const uint32_t g = v - 1, o = P.id_off[g], len = P.id_off[g + 1] - o - 1;
        if (len != n) continue;
        uint32_t i = 0;
        while (i < n && P.ids[o + i] == a[i]) ++i;
        if (i == n) return g;
      }
    }
    uint64_t sz;
    switch (ty) {
      case 'A': case 'c': case 'C': sz = 1; break;
      case 's': case 'S': sz = 2; break;
      case 'i': case 'I': case 'f': sz = 4; break;
      case 'Z': case 'H': {
        const uint8_t* z = a;
        while (z < end && *z) ++z;
        if (z >= end) { *bad = true; return none; }
        sz = (uint64_t)(z - a) + 1;
        break;
      }
      case 'B': {
        if (end - a < 5) { *bad = true; return none; }
        const uint8_t sub = a[0];
        const uint32_t cnt = (uint32_t)a[1] | ((uint32_t)a[2] << 8) | ((uint32_t)a[3] << 16) | ((uint32_t)a[4] << 24);
        uint32_t es;
        if (sub == 'c' || sub == 'C') es = 1;
        else if (sub == 's' || sub == 'S') es = 2;
        else if (sub == 'i' || sub == 'I' || sub == 'f') es = 4;
        else { *bad = true; return none; }
        sz = 5 + (uint64_t)cnt * es;
        break;
      }
      default: *bad = true; return none;
    }
    if ((uint64_t)(end - a) < sz) { *bad = true; return none; }
    a += sz;
  }
  return none;  // no RG field
}

// Records of one group are counted, and later scattered, with one atomic per distinct group in a warp (__match_any_sync): with
// few groups every record of a wave would otherwise hit the same counter, and same-address atomics serialise in L2.
__global__ void __launch_bounds__(kRgThreads) rg_tag_kernel(ReadGroupParams P) {
  const uint64_t n_rec = P.st->fatal ? 0 : P.st->wave_rec, rec_base = P.st->rec_base;
  const uint32_t lane = threadIdx.x & 31;
  uint32_t err = 0;
  for (uint64_t r0 = (uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); r0 < n_rec; r0 += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t r = r0 + lane;
    uint32_t g = kNoGroup;
    if (r < n_rec) {
      const uint8_t* p = P.d + (P.rec[r] & kRecOffMask);
      RecHeader h;
      if (load_record_header(p, P.n_ref, h) && (P.max_records == 0 || rec_base + r < P.max_records)) {
        const uint8_t* a = p + 36 + h.lname + 4 * (size_t)h.ncig + (h.lseq + 1) / 2 + h.lseq;
        bool bad = false;
        g = rg_lookup(a, p + 4 + (size_t)h.bs, P, &bad);
        if (bad) err = 1;
      }
      P.grp[r] = (uint16_t)g;
    }
    const uint32_t peers = __match_any_sync(0xFFFFFFFFu, g);
    if (g != kNoGroup && (int)lane == __ffs(peers) - 1) atomicAdd(&P.count[g], (uint32_t)__popc(peers));
  }
  if (err) P.res[R_ERR_RECORD] = 1;
}

// bucket g = [off_g, off_g + pad(count_g)), pad to a multiple of 32; the padding is filled with 0xFFFFFFFF
__global__ void __launch_bounds__(kRgScanThreads) rg_scan_kernel(ReadGroupParams P) {
  __shared__ uint32_t part[kRgScanThreads];
  const uint32_t n = P.n_groups + 1, per = (n + kRgScanThreads - 1) / kRgScanThreads;
  const uint32_t g0 = threadIdx.x * per, g1 = min(n, g0 + per);
  uint32_t s = 0;
  for (uint32_t g = g0; g < g1; ++g) s += (P.count[g] + 31u) & ~31u;
  part[threadIdx.x] = s;
  __syncthreads();
  for (uint32_t k = 1; k < kRgScanThreads; k <<= 1) {  // inclusive Hillis-Steele scan
    const uint32_t v = threadIdx.x >= k ? part[threadIdx.x - k] : 0u;
    __syncthreads();
    part[threadIdx.x] += v;
    __syncthreads();
  }
  uint32_t off = part[threadIdx.x] - s;
  for (uint32_t g = g0; g < g1; ++g) {
    const uint32_t c = P.count[g], padded = (c + 31u) & ~31u;
    P.cursor[g] = off;
    for (uint32_t i = c; i < padded; ++i) P.order[off + i] = 0xFFFFFFFFu;
    P.count[g] = 0;
    off += padded;
  }
  if (threadIdx.x == kRgScanThreads - 1) *P.total = part[kRgScanThreads - 1];
}

__global__ void __launch_bounds__(kRgThreads) rg_scatter_kernel(ReadGroupParams P) {
  const uint64_t n_rec = P.st->fatal ? 0 : P.st->wave_rec;
  const uint32_t lane = threadIdx.x & 31;
  for (uint64_t r0 = (uint64_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); r0 < n_rec; r0 += (uint64_t)gridDim.x * blockDim.x) {
    const uint64_t r = r0 + lane;
    const uint32_t g = r < n_rec ? (uint32_t)P.grp[r] : (uint32_t)kNoGroup;
    const uint32_t peers = __match_any_sync(0xFFFFFFFFu, g);
    const int leader = __ffs(peers) - 1;
    uint32_t base = 0;
    if (g != kNoGroup && (int)lane == leader) base = atomicAdd(&P.cursor[g], (uint32_t)__popc(peers));
    base = __shfl_sync(0xFFFFFFFFu, base, leader);
    if (g != kNoGroup) P.order[base + __popc(peers & ((1u << lane) - 1))] = (uint32_t)r;
  }
}

// Shared memory per warp: the 8-bit quality table of facets_kernel (kQualSmemPositions rows), 18 CIGAR-kind counters, and the
// TLEN and GC histograms as 8-bit counters, four to a word.  A record adds one to at most one bin of each, and the warp adds its
// histograms into the group's slice every kQualFlushSteps steps (224 records < 256) and when its group changes, like its quality
// table: no counter wraps or carries into the next byte.  Seven warps take 114 828 bytes, so two CTAs still fit on an SM.
constexpr uint32_t kRgTlenWords = (1025 + 3) / 4, kRgGcWords = (101 + 3) / 4;
constexpr uint32_t kRgWarpWords = 18 + kRgTlenWords + kRgGcWords;
__host__ __device__ inline size_t rg_facets_smem(uint32_t warps) { return (size_t)warps * (qual_table_bytes(kQualSmemPositions) + kRgWarpWords * 4); }

// One increment of bin `bin` (0xFFFFFFFF: none) per lane into a per-warp table of 8-bit counters packed in words: lanes with
// the same bin are counted by one shared-memory atomic of their leader.  Called by the whole warp.
__device__ __forceinline__ void byte_tally(uint32_t* words, uint32_t bin, uint32_t lane) {
  const uint32_t peers = __match_any_sync(0xFFFFFFFFu, bin);
  if (bin != 0xFFFFFFFFu && (int)lane == __ffs(peers) - 1) atomicAdd(&words[bin >> 2], (uint32_t)__popc(peers) << (8 * (bin & 3)));
}

// Adds a per-warp table of packed 8-bit counters into the u64 bins at `dst` and clears it
__device__ __forceinline__ void flush_byte_table(uint32_t* words, uint32_t n_words, uint64_t* dst, uint32_t lane) {
  for (uint32_t w = lane; w < n_words; w += 32) {
    const uint32_t v = words[w];
    if (!v) continue;
    words[w] = 0;
#pragma unroll
    for (uint32_t k = 0; k < 4; ++k) {
      const uint32_t c = (v >> (8 * k)) & 255u;
      if (c) atomicAdd((unsigned long long*)&dst[4 * w + k], (unsigned long long)c);
    }
  }
  __syncwarp();
}

__global__ void __launch_bounds__(kFacetThreads) rg_facets_kernel(ReadGroupParams P) {
  extern __shared__ uint32_t sm[];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  const uint32_t qtab_words = qual_table_bytes(kQualSmemPositions) / 4;
  uint32_t* my_qwords = sm + qtab_words * warp;
  uint8_t* my_qtab = reinterpret_cast<uint8_t*>(my_qwords);
  uint32_t* my_cig = sm + qtab_words * warps + kRgWarpWords * warp;
  uint32_t* my_tlen = my_cig + 18;
  uint32_t* my_gc = my_tlen + kRgTlenWords;
  for (uint32_t i = lane; i < qtab_words; i += 32) my_qwords[i] = 0;
  for (uint32_t i = lane; i < kRgWarpWords; i += 32) my_cig[i] = 0;
  __syncwarp();

  // contiguous step ranges per warp: a warp meets few group changes
  const uint64_t steps = *P.total / 32, n_warps = (uint64_t)gridDim.x * warps, w = (uint64_t)blockIdx.x * warps + warp;
  const uint64_t s0 = steps * w / n_warps, s1 = steps * (w + 1) / n_warps;
  uint32_t cur = 0xFFFFFFFFu, acc = 0, sum_gc = 0, sum_at = 0, sum_oth = 0, max_q = 0, since_flush = 0;
  uint32_t err_rec = 0;
  auto flush_tables = [&](uint32_t g) {  // the 8-bit tables: quality by position, TLEN and GC histograms
    flush_qual_table(my_qwords, kQualSmemPositions, (unsigned long long*)(P.qual + (uint64_t)g * P.rows * 94), lane);
    uint64_t* s = P.sums + (uint64_t)g * kGroupSums;
    flush_byte_table(my_tlen, kRgTlenWords, s + R_TLEN_HIST, lane);
    flush_byte_table(my_gc, kRgGcWords, s + R_GC_HIST, lane);
  };
  auto flush = [&](uint32_t g) {  // everything this warp holds for group g
    uint64_t* s = P.sums + (uint64_t)g * kGroupSums;
    if (acc && lane < 21) {
      const uint32_t slot = lane < 16 ? R_GENERAL + lane : lane == 16 ? R_TLEN_PROCESSED : lane == 17 ? R_TLEN_IGNORED : R_GC_REC + (lane - 18);
      atomicAdd((unsigned long long*)&s[slot], (unsigned long long)acc);
    }
    acc = 0;
    const uint32_t a = __reduce_add_sync(0xFFFFFFFFu, sum_gc), b = __reduce_add_sync(0xFFFFFFFFu, sum_at), c = __reduce_add_sync(0xFFFFFFFFu, sum_oth);
    sum_gc = sum_at = sum_oth = 0;
    if (lane == 0) {
      if (a) atomicAdd((unsigned long long*)&s[R_GC_NUC + 0], (unsigned long long)a);
      if (b) atomicAdd((unsigned long long*)&s[R_GC_NUC + 1], (unsigned long long)b);
      if (c) atomicAdd((unsigned long long*)&s[R_GC_NUC + 2], (unsigned long long)c);
      if (max_q) atomicMax((unsigned long long*)&P.qlen[g], (unsigned long long)max_q);
    }
    max_q = 0;
    __syncwarp();
    if (lane < 18) {
      const uint32_t v = my_cig[lane];
      if (v) { my_cig[lane] = 0; atomicAdd((unsigned long long*)&s[R_CIGAR + lane], (unsigned long long)v); }
    }
    flush_tables(g);
    since_flush = 0;
  };

  for (uint64_t step = s0; step < s1; ++step) {
    // ================= phase A: one record per lane =================
    const uint32_t ri = P.order[step * 32 + lane];
    bool on = ri != 0xFFFFFFFFu;
    const uint32_t g = __reduce_max_sync(0xFFFFFFFFu, on ? (uint32_t)P.grp[ri] : 0u);  // one group per step
    if (g != cur) {
      if (cur != 0xFFFFFFFFu) flush(cur);
      cur = g;
    }
    const uint8_t* p = P.d;
    uint64_t rv = 0;
    RecHeader h{};
    if (on) {
      rv = P.rec[ri];
      p = P.d + (rv & kRecOffMask);
      on = load_record_header(p, P.n_ref, h);  // rg_tag_kernel lists valid records only
    }
    const uint8_t* cig = p + 36 + h.lname;
    const uint8_t* seq = cig + 4 * (size_t)h.ncig;
    const uint32_t which = (h.f & 0x40) ? 0 : 9;
    if (on && h.ncig <= kShortCigar)
      for (uint32_t i = 0; i < h.ncig; ++i) {
        const uint32_t k = ld_u32_unaligned(cig + 4 * i) & 15;
        if (k <= 8) atomicAdd(&my_cig[which + k], 1u);
      }
    for (uint32_t todo = __ballot_sync(0xFFFFFFFFu, on && h.ncig > kShortCigar); todo; todo &= todo - 1) {
      const int j = __ffs(todo) - 1;
      const uint8_t* cj = reinterpret_cast<const uint8_t*>(__shfl_sync(0xFFFFFFFFu, (unsigned long long)cig, j));
      const uint32_t nj = __shfl_sync(0xFFFFFFFFu, h.ncig, j), wj = __shfl_sync(0xFFFFFFFFu, which, j);
      for (uint32_t i = lane; i < nj; i += 32) {
        const uint32_t k = ld_u32_unaligned(cj + 4 * i) & 15;
        if (k <= 8) atomicAdd(&my_cig[wj + k], 1u);
      }
    }
    uint32_t bits = 0, gc_off = 0;
    if (on) {
      bits = general_bits(h.f, h.ref, h.nref, h.mapq, err_rec) | tlen_bits(h.tlen) | gc_bits(h.f, h.lseq);
      if ((bits & (1u << 18)) && h.lseq > 100)
        gc_off = gc_window_offset(rv, P.blocks, P.st->carry_voff, P.headroom, P.out0, P.gc_seed, h.lseq);
    }
#pragma unroll
    for (int k = 0; k < 21; ++k) {
      const uint32_t m = __ballot_sync(0xFFFFFFFFu, (bits >> k) & 1u);
      if ((int)lane == k) acc += __popc(m);
    }
    uint32_t gc_bin = 0xFFFFFFFFu;
    if (bits & (1u << 18)) {
      uint32_t gc, at;
      gc_window_counts(seq, gc_off, &gc, &at);
      sum_gc += gc; sum_at += at; sum_oth += 100 - gc - at;
      gc_bin = gc;  // round(gc / 100 * 100) == gc
    }
    byte_tally(my_tlen, (bits & (1u << 16)) ? (uint32_t)h.tlen : 0xFFFFFFFFu, lane);
    byte_tally(my_gc, gc_bin, lane);

    // ================= phase B: one record per warp step: quality by position =================
    uint64_t* gq = P.qual + (uint64_t)g * P.rows * 94;
    for (uint32_t todo = __ballot_sync(0xFFFFFFFFu, on && h.lseq != 0); todo; todo &= todo - 1) {
      const int j = __ffs(todo) - 1;
      const uint8_t* sq = reinterpret_cast<const uint8_t*>(__shfl_sync(0xFFFFFFFFu, (unsigned long long)seq, j));
      const uint32_t ls = __shfl_sync(0xFFFFFFFFu, h.lseq, j);
      const uint8_t* ql = sq + (ls + 1) / 2;
      const uint32_t n_s = ls < kQualSmemPositions ? ls : kQualSmemPositions;
      const uint32_t n_g = ls < P.rows ? ls : P.rows;  // longer reads fail the run with NGSQ_E_QUAL_CAP
      bool any_real = false;
      for (uint32_t i = lane; i < ls; i += 32) {
        const uint32_t q = __ldg(ql + i);
        any_real |= q != 0xFF;
        if (q > 93) continue;
        if (i < n_s) { uint8_t* c = my_qtab + i * kQualRowBytes + q; *c = (uint8_t)(*c + 1); }
        else if (i < n_g) atomicAdd((unsigned long long*)&gq[(uint64_t)i * 94 + q], 1ull);
      }
      if (__any_sync(0xFFFFFFFFu, any_real)) max_q = ls > max_q ? ls : max_q;
    }
    __syncwarp();
    if (++since_flush == kQualFlushSteps) { flush_tables(g); since_flush = 0; }
  }
  if (cur != 0xFFFFFFFFu) flush(cur);
  if (err_rec) P.res[R_ERR_RECORD] = 1;
}

}  // namespace ngsq
