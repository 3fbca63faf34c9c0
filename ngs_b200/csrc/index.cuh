// K13 — BAI and CSI index build (`ngs index`, reference src/index/bam.rs:39-109 over noodles' BAI indexer; `samtools index
// -c` for CSI): per record, its (reference, bin, [beg, end)) key and start offset; per wave, the runs of records that share a
// (reference, bin), the order check, the per-reference counters and the per-window minimum offsets (16 kb windows for a BAI,
// 2^min_shift for a CSI).  The host (engine.cu, finish_index) turns the runs into chunks and writes the .bai or .csi bytes
// at ngsq_finish.  The contract is DESIGN.md section 4, "K13 index" and "K13 CSI".
//
// The per-record functions are NGSQ_HD: tools/index_model.cpp runs them on the CPU against the oracles
// (tests/cpp/bai_oracle.c, oracle_build_bai; tests/cpp/csi_oracle.c, oracle_build_csi; tests/test_index_model.py,
// test_index_model_csi.py).  GPU parity: tests/test_gpu_index.py, test_gpu_index_csi.py.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#include "recscan.cuh"
#endif

#ifndef NGSQ_HD
#if defined(__CUDACC__)
#define NGSQ_HD __host__ __device__ __forceinline__
#else
#define NGSQ_HD inline
#endif
#endif

namespace ngsq {

constexpr uint32_t kIxMetaBin = 37450;            // pseudo-bin of the per-reference metadata
constexpr uint64_t kIxMaxEnd = 1ull << 29;         // BAI addresses [0, 2^29); longer references need CSI
constexpr uint32_t kIxWindowShift = 14;            // 16 kb linear-index windows
constexpr uint64_t kIxUnplacedRun = ~0ull;         // run key of records that are in no bin
constexpr uint64_t kIxNoRun = ~1ull;               // run key "before the first record"
constexpr uint32_t kIxUnplacedRef = 0xFFFFFFFFu;   // IndexRun::ref of a run of unplaced records

// CSI binning (NGSQ_F_INDEX_CSI): windows of 2^min_shift bases, `depth` levels of bins below bin 0.  The bounds keep bin ids
// below 2^24 and a reference's window table (L >> min_shift) + 1 below 2^20 entries for any 32-bit length.
constexpr uint32_t kCsiMinShiftLo = 12, kCsiMinShiftHi = 24, kCsiDepthHi = 7;

enum : uint32_t {
  kIxBadRecord = 1,  // field overrun, CIGAR op > 8, reference id out of range
  kIxTooLong = 2,    // end > 2^29 (BAI) or 2^(min_shift + 3 depth) (CSI): not addressable
  kIxRunTable = 4,   // more runs than the wave's run table holds (sized by records: cannot happen)
  kIxOverflowList = 8,  // more records reach past their reference's window table than the overflow list holds
};

struct IndexKey {
  int32_t ref;        // reference id (-1 = none)
  int32_t pos;        // 0-based start as stored (-1 = none)
  uint32_t bin;       // reg2bin(beg, end) of a placed record
  uint32_t placed;    // ref >= 0 && pos >= 0: in a bin and in the linear index
  uint32_t unmapped;  // flag 0x4
  uint64_t beg, end;  // [beg, end) of a placed record
};

NGSQ_HD uint32_t ix_ld32(const uint8_t* p) {
  return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

// SAM spec section 5.3
NGSQ_HD uint32_t ix_reg2bin(uint64_t beg, uint64_t end) {
  --end;
  if (beg >> 14 == end >> 14) return (uint32_t)(((1u << 15) - 1) / 7 + (beg >> 14));
  if (beg >> 17 == end >> 17) return (uint32_t)(((1u << 12) - 1) / 7 + (beg >> 17));
  if (beg >> 20 == end >> 20) return (uint32_t)(((1u << 9) - 1) / 7 + (beg >> 20));
  if (beg >> 23 == end >> 23) return (uint32_t)(((1u << 6) - 1) / 7 + (beg >> 23));
  if (beg >> 26 == end >> 26) return (uint32_t)(((1u << 3) - 1) / 7 + (beg >> 26));
  return 0;
}

// CSIv1: hts_reg2bin, the generalised form of SAM 5.3 (at min_shift 14, depth 5 it is ix_reg2bin)
NGSQ_HD uint32_t ix_csi_reg2bin(uint64_t beg, uint64_t end, uint32_t min_shift, uint32_t depth) {
  --end;
  uint32_t s = min_shift, t = ((1u << 3 * depth) - 1) / 7;
  for (uint32_t l = depth; l > 0; --l, s += 3, t -= 1u << 3 * l)
    if (beg >> s == end >> s) return t + (uint32_t)(beg >> s);
  return 0;
}
// bins of a CSI: ids 0 .. n_bins - 1; the per-reference pseudo-bin is n_bins + 1 (37450 at depth 5, as in the BAI)
NGSQ_HD uint32_t ix_csi_n_bins(uint32_t depth) { return ((1u << 3 * (depth + 1)) - 1) / 7; }
NGSQ_HD uint64_t ix_csi_max_end(uint32_t min_shift, uint32_t depth) { return 1ull << (min_shift + 3 * depth); }
// first leaf window of a bin (htslib hts_bin_bot): the window whose filled minimum is the bin's loffset
NGSQ_HD uint64_t ix_csi_bin_bot(uint32_t bin, uint32_t depth) {
  uint32_t l = 0;
  for (uint32_t b = bin; b; b = (b - 1) >> 3) ++l;
  return (uint64_t)(bin - ((1u << 3 * l) - 1) / 7) << 3 * (depth - l);
}
// samtools index -c: the smallest depth n with max_len + 256 <= 2^(min_shift + 3n)
NGSQ_HD uint32_t ix_csi_default_depth(uint64_t max_len, uint32_t min_shift) {
  uint32_t n = 0;
  for (uint64_t s = 1ull << min_shift; max_len + 256 > s; s <<= 3) ++n;
  return n;
}

// Header of the record at `rec` (its block_size first): fills ref / pos / unmapped and the CIGAR's place; 0 or kIxBadRecord.
NGSQ_HD uint32_t index_header(const uint8_t* rec, int32_t n_ref, IndexKey* k, uint32_t* ncig, const uint8_t** cig) {
  const uint32_t bs = ix_ld32(rec);
  k->ref = (int32_t)ix_ld32(rec + 4);
  k->pos = (int32_t)ix_ld32(rec + 8);
  const uint32_t w3 = ix_ld32(rec + 12), w4 = ix_ld32(rec + 16), lseq = ix_ld32(rec + 20);
  const int32_t nref = (int32_t)ix_ld32(rec + 24);
  const uint32_t lname = w3 & 255;
  *ncig = w4 & 0xFFFF;
  *cig = rec + 36 + lname;
  k->unmapped = (w4 >> 16) & 0x4u ? 1u : 0u;
  k->placed = 0;
  k->bin = 0;
  k->beg = k->end = 0;
  if (bs < 32 || 32ull + lname + 4ull * *ncig + (lseq + 1ull) / 2 + lseq > bs) return kIxBadRecord;
  if (k->ref < -1 || k->ref >= n_ref || nref < -1 || nref >= n_ref) return kIxBadRecord;
  return 0;
}

// Reference span of CIGAR ops [i0, n) in steps of `step` (M D N = X, utils/cigar.rs:6-11); 0 or kIxBadRecord (op > 8).
NGSQ_HD uint32_t index_cigar_span(const uint8_t* cig, uint32_t i0, uint32_t n, uint32_t step, uint64_t* span) {
  uint64_t s = 0;
  uint32_t bad = 0;
  for (uint32_t i = i0; i < n; i += step) {
    const uint32_t op = ix_ld32(cig + 4 * i), kind = op & 15;
    if (kind > 8) bad = kIxBadRecord;
    else if ((0x18Du >> kind) & 1u) s += op >> 4;
  }
  *span = s;
  return bad;
}

// Completes the key once the span is known: [beg, end) with a zero span counted as 1, and the bin.  0 or kIxTooLong.
NGSQ_HD uint32_t index_finish_key(IndexKey* k, uint64_t span) {
  if (k->ref < 0 || k->pos < 0) return 0;
  k->placed = 1;
  k->beg = (uint64_t)k->pos;
  k->end = k->beg + (span ? span : 1);
  if (k->end > kIxMaxEnd) { k->placed = 0; return kIxTooLong; }
  k->bin = ix_reg2bin(k->beg, k->end);
  return 0;
}

// The same for a CSI of the given binning.  0 or kIxTooLong (end > 2^(min_shift + 3 depth)).
NGSQ_HD uint32_t index_finish_key_csi(IndexKey* k, uint64_t span, uint32_t min_shift, uint32_t depth) {
  if (k->ref < 0 || k->pos < 0) return 0;
  k->placed = 1;
  k->beg = (uint64_t)k->pos;
  k->end = k->beg + (span ? span : 1);
  if (k->end > ix_csi_max_end(min_shift, depth)) { k->placed = 0; return kIxTooLong; }
  k->bin = ix_csi_reg2bin(k->beg, k->end, min_shift, depth);
  return 0;
}

// The whole key of one record, serially (the host model; the kernel splits the CIGAR walk over a warp for long CIGARs).
// csi = 0: the BAI key; otherwise the CSI key at (min_shift, depth).
NGSQ_HD uint32_t index_record(const uint8_t* rec, int32_t n_ref, IndexKey* k, bool csi = false, uint32_t min_shift = 0, uint32_t depth = 0) {
  uint32_t ncig;
  const uint8_t* cig;
  uint32_t bad = index_header(rec, n_ref, k, &ncig, &cig);
  if (bad) return bad;
  uint64_t span;
  if ((bad = index_cigar_span(cig, 0, ncig, 1, &span))) return bad;
  return csi ? index_finish_key_csi(k, span, min_shift, depth) : index_finish_key(k, span);
}

// Windows [lo, hi] a placed record touches, of 2^shift bases (kIxWindowShift: the BAI's linear index).
NGSQ_HD void index_windows(const IndexKey& k, uint32_t* lo, uint32_t* hi, uint32_t shift = kIxWindowShift) {
  *lo = (uint32_t)(k.beg >> shift);
  *hi = (uint32_t)((k.end - 1) >> shift);
}

// Runs: consecutive records with equal keys share a chunk.  Unplaced records share one key: they end a chunk, join none.
NGSQ_HD uint64_t index_run_key(const IndexKey& k) { return k.placed ? ((uint64_t)(uint32_t)k.ref << 32) | k.bin : kIxUnplacedRun; }
// Order: placed records must be non-decreasing in (ref, pos) and none may follow a ref = -1 record.  Records with ref >= 0 and
// pos = -1 constrain nothing.
NGSQ_HD bool index_constrains(const IndexKey& k) { return k.placed || k.ref < 0; }
NGSQ_HD uint64_t index_order_key(const IndexKey& k) { return k.ref < 0 ? ~0ull : ((uint64_t)(uint32_t)k.ref << 32) | (uint32_t)k.pos; }

// One entry of the run table (and of the BAI's overflow list, whose `bin` holds window lo | hi << 16).
struct IndexRun {
  uint64_t voff;  // virtual offset of the run's first record; the run ends where the next one starts
  uint32_t ref;   // kIxUnplacedRef for unplaced records
  uint32_t bin;
};
// One entry of the CSI's overflow list: windows [lo, hi] of a record past its reference's table (a CSI reference may have
// more than 2^16 windows)
struct IndexOvf {
  uint64_t voff;
  uint32_t ref, lo, hi, pad;
};

#if defined(__CUDACC__)

// What links two waves, double-buffered by the parity of the indexed wave: the kernel of wave j reads carry[j & 1] and its
// last record writes carry[(j + 1) & 1].
struct IndexCarry {
  uint64_t run_key;    // of the last record
  uint64_t order_key;  // of the last record that constrains the order (0 = none yet)
};

struct IndexState {
  // NGSQ_F_INDEX_PART: order key and virtual offset of the part's first placed record (~0 = none), the two halves of one
  // 128-bit word with the offset high, so that a 128-bit minimum takes the first record with its key
  alignas(16) unsigned long long first_key;
  unsigned long long first_voff;
  IndexCarry carry[2];
  unsigned long long n_runs[2];     // entries in the run table of slot j & 1 (zeroed before the wave's kernel)
  unsigned long long n_no_coor;     // unplaced records
  unsigned long long unsorted_voff; // smallest virtual offset of a placed record out of order (~0 = none)
  unsigned long long n_ovf;         // overflow-list entries
  unsigned int err;                 // kIx* bits
};

struct IndexParams {
  const uint8_t* d;         // base of the wave's slot
  const uint64_t* rec;      // record table of the wave (recscan.cuh)
  const RunState* st;       // wave_rec, carry_voff, fatal
  const BlockDesc* blocks;  // the wave's blocks (file offsets for virtual offsets)
  uint32_t headroom;
  uint32_t par;             // parity of the indexed wave
  uint64_t out0;
  int32_t n_ref;
  IndexState* S;
  IndexRun* runs;           // this wave's run table
  uint64_t runs_cap;
  void* ovf;                // whole run: records whose windows reach past their reference's table (IndexRun for a BAI,
                            // IndexOvf for a CSI)
  uint64_t ovf_cap;
  const uint64_t* win_base; // per reference: first entry in win
  const uint32_t* win_n;    // per reference: windows in the table ((L >> shift) + 1)
  unsigned long long* win;  // smallest start offset per window (~0 = untouched)
  unsigned int* max_win;    // per reference: largest window touched
  unsigned long long* counts;  // per reference: mapped, unmapped
  uint32_t part;            // NGSQ_F_INDEX_PART: also record the first placed record (IndexState::first_key / first_voff)
  uint32_t min_shift, depth;  // CSI binning (index_kernel<true>)
};

// 128-bit minimum of (voff, key) into S->first_key / first_voff.  A torn read of the current value only costs a failed CAS:
// the offset half never grows, and no two records share an offset.
__device__ __forceinline__ void index_first_min(IndexState* S, uint64_t voff, uint64_t key) {
  unsigned __int128* p = reinterpret_cast<unsigned __int128*>(&S->first_key);
  const unsigned __int128 v = ((unsigned __int128)voff << 64) | key;
  const volatile unsigned long long* h = &S->first_key;
  unsigned __int128 o = ((unsigned __int128)h[1] << 64) | h[0];
  while (v < o) {
    const unsigned __int128 r = atomicCAS(p, o, v);
    if (r == o) break;
    o = r;
  }
}

constexpr int kIndexThreads = 256;

// Virtual offset of record r of the wave: its block's file offset and its offset in that block (the carried record: the one
// the previous wave recorded), as facets.cuh computes it for the GC window.
__device__ __forceinline__ uint64_t index_voff(const IndexParams& P, uint64_t rv) {
  const uint32_t t = (uint32_t)(rv >> 40);
  if (!t) return P.st->carry_voff;
  const BlockDesc& bd = P.blocks[t - 1];
  return (bd.coff << 16) | ((rv & kRecOffMask) - P.headroom - (bd.out_off - P.out0));
}

// Warp steps of 31 records: lane l holds record r0 - 1 + l, so every lane but 0 finds its predecessor's key in lane l - 1;
// lane 0 holds the previous step's last record (or, for record 0 of the wave, the carry of the previous wave).
// kCsi = false: the BAI (bins of SAM 5.3, 16 kb windows, ends up to 2^29); true: the CSI binning of P.min_shift / P.depth.
// The two differ only in constexpr branches, so the BAI instance is the kernel it was before CSI existed.
template <bool kCsi>
__global__ void __launch_bounds__(kIndexThreads) index_kernel(IndexParams P) {
  const uint32_t lane = threadIdx.x & 31;
  const uint64_t n = P.st->fatal ? 0 : P.st->wave_rec;
  const IndexCarry cin = P.S->carry[P.par];
  if (n == 0) {
    if (blockIdx.x == 0 && threadIdx.x == 0) P.S->carry[P.par ^ 1] = cin;
    return;
  }
  const uint64_t warp = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
  uint32_t err = 0;
  uint64_t no_coor = 0;
  unsigned long long unsorted = ~0ull;
  for (uint64_t r0 = warp * 31; r0 < n; r0 += n_warps * 31) {
    const int64_t r = (int64_t)r0 - 1 + (int64_t)lane;
    const bool have = r >= 0 && (uint64_t)r < n;
    const bool own = lane > 0 && have;
    IndexKey k{};
    k.ref = -1;
    k.pos = -1;
    uint32_t bad = 0, ncig = 0;
    const uint8_t* cig = nullptr;
    uint64_t voff = 0, span = 0;
    if (have) {
      const uint64_t rv = P.rec[r];
      voff = index_voff(P, rv);
      bad = index_header(P.d + (rv & kRecOffMask), P.n_ref, &k, &ncig, &cig);
      if (!bad && ncig <= 8) bad = index_cigar_span(cig, 0, ncig, 1, &span);
    }
    // long CIGARs (long reads): the whole warp strides over one record's ops
    for (uint32_t todo = __ballot_sync(0xFFFFFFFFu, have && !bad && ncig > 8); todo; todo &= todo - 1) {
      const int j = __ffs(todo) - 1;
      const uint8_t* cj = reinterpret_cast<const uint8_t*>(__shfl_sync(0xFFFFFFFFu, (unsigned long long)cig, j));
      const uint32_t nj = __shfl_sync(0xFFFFFFFFu, ncig, j);
      uint64_t sp;
      const uint32_t b = index_cigar_span(cj, lane, nj, 32, &sp);
      for (int o = 16; o; o >>= 1) sp += __shfl_xor_sync(0xFFFFFFFFu, sp, o);  // 64-bit: the sum may pass 2^32 (then end > 2^29)
      const bool any_bad = __any_sync(0xFFFFFFFFu, b);
      if ((int)lane == j) { span = sp; if (any_bad) bad = kIxBadRecord; }
    }
    if (have && !bad) {
      if constexpr (kCsi) bad = index_finish_key_csi(&k, span, P.min_shift, P.depth);
      else bad = index_finish_key(&k, span);
    }
    if (bad) { k.ref = -1; k.pos = -1; k.placed = 0; if (own) err |= bad; }

    // ---- runs: a record starts one when its key differs from its predecessor's
    const uint64_t rk = have ? index_run_key(k) : (r < 0 ? cin.run_key : 0);
    const uint64_t prev_rk = __shfl_up_sync(0xFFFFFFFFu, rk, 1);
    const bool start = own && rk != prev_rk;

    // ---- order: a placed record against the last record before it that constrains the order
    const bool cons = have && index_constrains(k);
    const uint32_t cm = __ballot_sync(0xFFFFFFFFu, cons);
    uint64_t v0 = cons ? index_order_key(k) : 0;
    if (lane == 0 && !cons) {
      // the record before lane 0 that constrains: walk back over records with ref >= 0, pos = -1 (each is walked over by one
      // warp at most, the one whose lane 0 follows it), headers only
      v0 = cin.order_key;
      for (int64_t q = r - 1; q >= 0; --q) {
        const uint8_t* p = P.d + (P.rec[q] & kRecOffMask);
        const int32_t qref = (int32_t)ix_ld32(p + 4), qpos = (int32_t)ix_ld32(p + 8);
        if (qref < 0) { v0 = ~0ull; break; }
        if (qpos >= 0) { v0 = ((uint64_t)(uint32_t)qref << 32) | (uint32_t)qpos; break; }
      }
    }
    const uint32_t upto_mask = cm & (lane == 31 ? 0xFFFFFFFFu : ((2u << lane) - 1u));
    const uint64_t upto = __shfl_sync(0xFFFFFFFFu, v0, upto_mask ? 31 - __clz(upto_mask) : 0);
    const uint64_t pred = __shfl_up_sync(0xFFFFFFFFu, upto, 1);
    if (own && k.placed && index_order_key(k) < pred) unsorted = voff < unsorted ? voff : unsorted;
    if (own && (uint64_t)r == n - 1) P.S->carry[P.par ^ 1] = IndexCarry{rk, upto};

    // ---- run table: one ticket per warp
    const uint32_t sm = __ballot_sync(0xFFFFFFFFu, start);
    if (sm) {
      const int leader = __ffs(sm) - 1;
      unsigned long long base = 0;
      if ((int)lane == leader) base = atomicAdd(&P.S->n_runs[P.par], (unsigned long long)__popc(sm));
      base = __shfl_sync(0xFFFFFFFFu, base, leader);
      if (start) {
        const uint64_t idx = base + __popc(sm & ((1u << lane) - 1));
        if (idx < P.runs_cap) P.runs[idx] = IndexRun{voff, k.placed ? (uint32_t)k.ref : kIxUnplacedRef, k.placed ? k.bin : 0u};
        else err |= kIxRunTable;
      }
    }

    // ---- counters
    const bool pl = own && k.placed;
    no_coor += __popc(__ballot_sync(0xFFFFFFFFu, own && !k.placed && !bad));
    const uint32_t pm = __ballot_sync(0xFFFFFFFFu, pl);
    if (P.part && pm && (int)lane == __ffs(pm) - 1) index_first_min(P.S, voff, index_order_key(k));  // the warp's first in file order
    uint32_t w_lo = 0, w_hi = 0, nw = 0;
    if (pl) {
      if constexpr (kCsi) index_windows(k, &w_lo, &w_hi, P.min_shift);
      else index_windows(k, &w_lo, &w_hi);
      nw = P.win_n[k.ref];
      const uint32_t cslot = 2u * (uint32_t)k.ref + k.unmapped;
      const uint32_t peers = __match_any_sync(pm, cslot);
      if ((int)lane == __ffs(peers) - 1) atomicAdd(&P.counts[cslot], (unsigned long long)__popc(peers));
      const uint32_t rpeers = __match_any_sync(pm, (uint32_t)k.ref);
      const uint32_t mx = __reduce_max_sync(rpeers, w_hi);
      if ((int)lane == __ffs(rpeers) - 1) atomicMax(&P.max_win[k.ref], mx);
    }
    // ---- linear index: one atomicMin per distinct window per warp (lanes are in file order: the lowest lane has the
    // smallest offset); long and spliced reads loop over all their windows
    const bool tab = pl && w_lo < nw;
    const uint32_t t_hi = tab ? (w_hi < nw ? w_hi : nw - 1) : 0;
    const uint64_t wb = pl ? P.win_base[k.ref] : 0;
    for (uint32_t i = 0;; ++i) {
      const bool act = tab && w_lo + i <= t_hi;
      const uint32_t am = __ballot_sync(0xFFFFFFFFu, act);
      if (!am) break;
      if (act) {
        const unsigned long long addr = wb + w_lo + i;
        const uint32_t peers = __match_any_sync(am, addr);
        if ((int)lane == __ffs(peers) - 1) atomicMin(&P.win[addr], (unsigned long long)voff);
      }
    }
    // windows past the table: reads that overhang the end of their reference
    const bool over = pl && w_hi >= nw;
    const uint32_t om = __ballot_sync(0xFFFFFFFFu, over);
    if (om) {
      const int leader = __ffs(om) - 1;
      unsigned long long base = 0;
      if ((int)lane == leader) base = atomicAdd(&P.S->n_ovf, (unsigned long long)__popc(om));
      base = __shfl_sync(0xFFFFFFFFu, base, leader);
      if (over) {
        const uint64_t idx = base + __popc(om & ((1u << lane) - 1));
        const uint32_t lo = w_lo > nw ? w_lo : nw;
        if (idx < P.ovf_cap) {
          if constexpr (kCsi) static_cast<IndexOvf*>(P.ovf)[idx] = IndexOvf{voff, (uint32_t)k.ref, lo, w_hi, 0u};
          else static_cast<IndexRun*>(P.ovf)[idx] = IndexRun{voff, (uint32_t)k.ref, lo | (w_hi << 16)};
        } else err |= kIxOverflowList;
      }
    }
  }
  if (lane == 0 && no_coor) atomicAdd(&P.S->n_no_coor, (unsigned long long)no_coor);
  if (unsorted != ~0ull) atomicMin(&P.S->unsorted_voff, unsorted);
  if (err) atomicOr(&P.S->err, err);
}

#endif  // __CUDACC__

}  // namespace ngsq
