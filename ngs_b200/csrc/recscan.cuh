// K3 — record-boundary scan over one WAVE of the inflated byte stream (reference: the record framing
// that bam::Reader::records / query perform one record at a time, src/qc/command.rs:305, :369-377).
//
// The engine streams the file in waves (the BGZF blocks of one inflate launch).  A wave's inflated bytes
// sit in one of two recycled slots:
//
//     slot:   [ headroom H ................ | block 0 | block 1 | ... | block n-1 ]
//                          [ carry ]^H                                          ^wave_end
//
// BAM records form a linked list (next = off + 4 + block_size) that ignores BGZF blocks and waves.  The
// record that is still open at the end of wave k (the "carry": from its first byte to the end of the wave)
// is copied in front of wave k+1's first block, so every record is contiguous in exactly one slot and no
// kernel needs carry-over logic.  Everything that links two waves lives in RunState on the DEVICE: a wave is
// enqueued without any host round trip (the host thread keeps feeding the copy engine).
//
// Per wave the chain is broken per BGZF block:
//   1. find_first  — one warp per block tests its first bytes, 32 candidate offsets at a time, for a
//                    plausible record header confirmed by a 3-record chain;
//   2. walk<count> — one thread per block (plus one for the carried record) walks from its first record to
//                    the block end, counts records and CHECKS CLOSURE: the walk must land exactly on the
//                    first record found for the block it lands in, blocks it jumps over must claim none,
//                    and exactly one walk reaches the end of the wave (it names the next carry);
//   3. check_landed, then chain_fix: a closure failure makes ONE thread rebuild the wave's first-record
//                    table serially (correct by construction) and the closure pass is repeated — a false
//                    positive of step 1 can never change results;
//   4. scan_counts — exclusive scan of the counts + the wave's commit (record count, next carry, errors);
//   5. walk<emit>  — same walk, writes rec[i] = offset in the slot | (block + 1) << 40 (0 = the carried record).
// find_record_kernel serves ngsq_find_record (record anchors of a file without an index) with the same plausibility test.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "inflate_lane.cuh"  // BlockDesc

namespace ngsq {

constexpr uint32_t kNoFirst = 0xFFFFFFFFu;
constexpr uint32_t kMaxRecordBytes = 1u << 28;
constexpr uint64_t kNoCarry = ~0ull;
constexpr uint64_t kRecOffMask = (1ull << 40) - 1;  // record table entry: slot offset | (block + 1) << 40

// fatal conditions (RunState::fatal bits): once one is set, the remaining kernels of the run do nothing
enum : uint32_t {
  kFatalInflate = 1u,    // a BGZF block failed to inflate
  kFatalChain = 2u,      // the record chain does not close (even after the serial rebuild)
  kFatalTruncated = 4u,  // the chain runs past the end of the data
  kFatalBadRecord = 8u,  // implausible block_size / l_seq on a verified chain
  kFatalCarry = 16u,     // a record does not fit the slot's headroom
  kFatalRecTable = 32u,  // more records than the wave's table holds (sized by bytes / 36: cannot happen)
};

struct RunState {
  // ---- whole run (sticky) ----
  uint32_t fatal;
  uint32_t crc_bad;
  unsigned long long bad_block;  // min over failed blocks of (global index << 8 | inflate status)
  uint32_t max_lseq;
  uint32_t qual_overflow;   // longest read whose qualities did not fit the global table (0 = none)
  uint32_t end_reached;     // the shard's end offset was met in an EARLIER wave: nothing left that this shard owns
  uint32_t end_pending;     // ... met in the current wave (becomes end_reached at the next wave_begin)
  uint64_t rec_base;        // records emitted by earlier waves
  uint64_t wave_rec;        // records of the current wave (adjacent to rec_base: the host's progress probe copies both)
  uint32_t waves, pad2;
  // the carry the last committed wave hands to the next one (written by scan_counts_kernel, consumed by wave_begin_kernel)
  uint64_t cn_voff;         // virtual offset of the record
  uint64_t cn_src;          // slot offset of its first byte in the slot of the wave that committed it
  uint32_t cn_len, pad3;    // bytes (0: the next wave starts on a record boundary)
  // ---- current wave ----
  uint64_t carry_voff;      // virtual offset of the record carried INTO this wave
  uint32_t carry_len, pad4; // its bytes in front of the wave's first block
  uint32_t wave_chain, wave_bad, wave_trunc, redo, wave_end_reached;
  uint32_t wave_long;       // reads longer than the facet kernel's shared-memory quality tables (facets.cuh: LongRead list)
  uint64_t next_carry;      // slot offset where the walk that reached the end of the wave stopped
  uint64_t next_carry_voff;
  // ---- pass-2 `-n` (cov_n.cuh): query-yielded records so far, reference id + 1 of the last one ----
  uint64_t cov_yielded;
  uint32_t cov_last_ref, pad1;
};

struct WaveParams {
  const uint8_t* d;         // slot base
  uint64_t out0;            // offset of the wave's first block in the whole inflated stream
  const BlockDesc* blocks;  // the wave's blocks; block b sits at d + headroom + (out_off - out0)
  const uint32_t* status;   // inflate verdict per block
  uint32_t n_blocks;
  uint32_t first_global;    // global index of blocks[0]
  uint32_t headroom;
  uint32_t first_wave;      // the shard's first record lies in this wave, at start_off
  uint32_t final_wave;      // nothing follows: a record that runs past wave_end is a truncation
  int32_t n_ref;
  uint64_t wave_end;        // headroom + inflated bytes of the wave
  uint64_t start_off;       // slot offset of the shard's first record (first_wave only)
  uint64_t end_off;         // slot offset of the first record the shard does NOT own; ~0 if it is not in this wave
  uint64_t rec_cap;
  RunState* st;
  uint32_t *first, *landed;  // [n_blocks]
  uint32_t* count;           // [n_blocks + 1]; index 0 = the carried record, t = block t - 1
  uint64_t* base;            // likewise
  uint64_t* rec;
};

__device__ __forceinline__ uint32_t ld_u32_unaligned(const uint8_t* p) {
  uintptr_t a = reinterpret_cast<uintptr_t>(p);
  const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~uintptr_t(3));
  uint32_t sh = (uint32_t)(a & 3) * 8;
  uint32_t lo = w[0];
  if (sh == 0) return lo;
  uint32_t hi = w[1];
  return __funnelshift_r(lo, hi, sh);
}

__device__ __forceinline__ uint64_t wave_root(const WaveParams& W) {
  return W.first_wave ? W.start_off : (uint64_t)W.headroom - W.st->carry_len;  // carry_len is 0 in the first wave
}
__device__ __forceinline__ uint64_t block_lo(const WaveParams& W, uint32_t b) { return W.headroom + (W.blocks[b].out_off - W.out0); }
__device__ __forceinline__ bool wave_dead(const RunState* st) { return st->fatal || st->end_reached; }

// Header plausibility of a record starting at slot offset `off`; [.., d_end) is the data a record of this wave may
// use.  Returns the offset of the next record, 0 when implausible; with open_end (more data follows this wave) a
// record that runs past d_end is accepted on its header alone and d_end is returned.
__device__ __forceinline__ uint64_t plausible(const uint8_t* d, uint64_t off, uint64_t d_end, int32_t n_ref, bool open_end) {
  if (off + 36 > d_end) return 0;
  const uint8_t* p = d + off;
  uint32_t bs = ld_u32_unaligned(p);
  if (bs < 34 || bs > kMaxRecordBytes) return 0;
  const bool past = off + 4 + bs > d_end;
  if (past && !open_end) return 0;
  int32_t ref = (int32_t)ld_u32_unaligned(p + 4);
  int32_t pos = (int32_t)ld_u32_unaligned(p + 8);
  uint32_t w3 = ld_u32_unaligned(p + 12);  // l_read_name, mapq, bin
  uint32_t w4 = ld_u32_unaligned(p + 16);  // n_cigar, flag
  uint32_t lseq = ld_u32_unaligned(p + 20);
  int32_t nref = (int32_t)ld_u32_unaligned(p + 24);
  int32_t npos = (int32_t)ld_u32_unaligned(p + 28);
  uint32_t lname = w3 & 255, ncig = w4 & 0xFFFF;
  if (ref < -1 || ref >= n_ref || nref < -1 || nref >= n_ref) return 0;
  if (pos < -1 || npos < -1 || lname < 2) return 0;
  uint64_t need = 32ull + lname + 4ull * ncig + (lseq + 1ull) / 2 + lseq;
  if (need > bs) return 0;
  if (off + 36 + lname <= d_end && p[36 + lname - 1] != 0) return 0;  // read name is NUL-terminated
  if (off + 37 <= d_end) {
    uint8_t c0 = p[36];
    if (c0 < 33 || c0 > 126) return 0;
  }
  return past ? d_end : off + 4 + bs;
}

// Start of a wave (one CTA): brings the carry in front of the wave's first block and opens the per-wave state.
// prev = base of the slot that holds the previous wave.
__global__ void __launch_bounds__(1024) wave_begin_kernel(RunState* st, uint8_t* cur, const uint8_t* prev, uint32_t headroom, uint32_t first_wave) {
  const uint32_t n = first_wave ? 0u : st->cn_len;
  if (!st->fatal && prev && n) {
    const uint8_t* src = prev + st->cn_src;
    uint8_t* dst = cur + headroom - n;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) dst[i] = src[i];
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    st->carry_len = n;
    st->carry_voff = st->cn_voff;
    if (st->end_pending) st->end_reached = 1;
    st->rec_base += st->wave_rec;
    st->wave_rec = 0;
    st->wave_chain = st->wave_bad = st->wave_trunc = st->redo = st->wave_end_reached = st->wave_long = 0;
    st->next_carry = kNoCarry;
    st->waves++;
  }
}

// Waves outside the shard's range are inflated (and CRC-checked) like the rest; only their verdicts are folded.
__global__ void status_fold_kernel(const uint32_t* __restrict__ status, uint32_t n_blocks, uint32_t first_global, RunState* st) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= n_blocks || !status[b]) return;
  atomicOr(&st->fatal, kFatalInflate);
  atomicMin(&st->bad_block, ((unsigned long long)(first_global + b) << 8) | status[b]);
}

// first[b] for every block of the wave; also folds the inflate verdicts into the run state.
__global__ void find_first_kernel(WaveParams W) {
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const uint32_t lane = threadIdx.x & 31;
  if (warp >= W.n_blocks) return;
  RunState* st = W.st;
  if (lane == 0 && W.status[warp]) {
    atomicOr(&st->fatal, kFatalInflate);
    atomicMin(&st->bad_block, ((unsigned long long)(W.first_global + warp) << 8) | W.status[warp]);
  }
  if ((st->fatal & ~kFatalInflate) || st->end_reached) { if (lane == 0) W.first[warp] = kNoFirst; return; }
  const uint64_t root = wave_root(W);
  const uint64_t lo = block_lo(W, warp), hi = lo + W.blocks[warp].isize;
  const bool end_here = W.end_off <= W.wave_end;
  const uint64_t d_end = end_here ? W.end_off : W.wave_end;
  const bool open_end = !end_here && !W.final_wave;
  uint32_t res = kNoFirst;
  if (root >= hi || lo >= d_end) {
    // blocks wholly before the shard's first record or behind its end hold nothing we own
  } else if (root >= lo) {
    res = (uint32_t)(root - lo);  // the root block: exact, never speculated
  } else {
    for (uint64_t base = lo; base < hi; base += 32) {
      uint64_t c = base + lane;
      // cheap necessary condition first: a block that lies wholly inside a long read has no record start, and all of its
      // 65536 offsets would otherwise pay for the full header + chain test (configs[3]: 272 ms of a 1757 ms step)
      bool pre = false;
      if (c < hi && c + 36 <= d_end) {
        const uint32_t bs0 = ld_u32_unaligned(W.d + c);
        const int32_t ref0 = (int32_t)ld_u32_unaligned(W.d + c + 4);
        pre = bs0 >= 34 && bs0 <= kMaxRecordBytes && ref0 >= -1 && ref0 < W.n_ref && (open_end || c + 4 + bs0 <= d_end);
      }
      if (!__any_sync(0xFFFFFFFFu, pre)) continue;
      bool ok = false;
      if (pre) {
        uint64_t n1 = plausible(W.d, c, d_end, W.n_ref, open_end);
        if (n1) {
          ok = true;
          // confirm with up to two further records when they fit in the data
          uint64_t n2 = n1 + 36 <= d_end ? plausible(W.d, n1, d_end, W.n_ref, open_end) : n1;
          if (!n2) ok = false;
          else if (n2 != n1) {
            uint64_t n3 = n2 + 36 <= d_end ? plausible(W.d, n2, d_end, W.n_ref, open_end) : n2;
            if (!n3) ok = false;
          }
        }
      }
      uint32_t m = __ballot_sync(0xFFFFFFFFu, ok);
      if (m) {
        res = (uint32_t)(base - lo) + (__ffs(m) - 1);
        break;
      }
    }
  }
  if (lane == 0) W.first[warp] = res;
}

// ngsq_find_record: one thread per offset of an inflated window [0, n) (grid-stride, so a thread's offsets only grow).  An
// offset passes when a chain of plausible records starts there and runs to the end of the window (the last record may run
// past it; a tail too short for a header is not judged).  *best = the smallest passing offset (~0 = none).
__global__ void find_record_kernel(const uint8_t* __restrict__ d, uint64_t n, int32_t n_ref, unsigned long long* best) {
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
  for (uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; c + 36 <= n; c += stride) {
    if (c >= *(volatile unsigned long long*)best) return;
    uint64_t off = c;
    bool ok = true;
    while (off + 36 <= n) {
      const uint64_t nx = plausible(d, off, n, n_ref, true);
      if (!nx) { ok = false; break; }
      off = nx;
    }
    if (ok) { atomicMin(best, (unsigned long long)c); return; }
  }
}

// the walk that reaches the end of the wave names the next carry; two different claims = two chains = closure failure
__device__ __forceinline__ void claim_carry(RunState* st, uint64_t off, uint64_t voff, bool set_voff) {
  const unsigned long long old = atomicCAS((unsigned long long*)&st->next_carry, (unsigned long long)kNoCarry, (unsigned long long)off);
  if (old == kNoCarry) { if (set_voff) st->next_carry_voff = voff; }
  else if (old != off) atomicAdd(&st->wave_chain, 1u);
}

// Thread 0 walks the carried record, thread t > 0 block t - 1.  EMIT=false: count + closure; EMIT=true: offset table.
// REDO: the second closure pass, which runs only after chain_fix_kernel rebuilt first[].
template <bool EMIT, bool REDO>
__global__ void walk_kernel(WaveParams W) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t > W.n_blocks) return;
  RunState* st = W.st;
  if (REDO && !st->redo) return;
  if (wave_dead(st)) { if (!EMIT) W.count[t] = 0; return; }
  uint64_t lo, hi, off;
  if (t == 0) {
    const uint32_t cl = st->carry_len;
    if (!cl) { if (!EMIT) W.count[0] = 0; return; }
    lo = (uint64_t)W.headroom - cl;
    hi = W.headroom;
    off = lo;
  } else {
    const uint32_t f = W.first[t - 1];
    if (f == kNoFirst) { if (!EMIT) W.count[t] = 0; return; }
    lo = block_lo(W, t - 1);
    hi = lo + W.blocks[t - 1].isize;
    off = lo + f;
  }
  const uint64_t stop = hi < W.end_off ? hi : W.end_off;
  uint32_t n = 0, max_lseq = 0;
  const uint64_t w = EMIT ? W.base[t] : 0;
  bool open = false;
  while (off < stop) {
    uint32_t bs = 0;
    const bool hdr_fits = off + 36 <= W.wave_end;
    if (hdr_fits) {
      bs = ld_u32_unaligned(W.d + off);
      if (bs < 32 || bs > kMaxRecordBytes) { if (!EMIT) atomicAdd(&st->wave_bad, 1u); open = true; break; }
    }
    if (!hdr_fits || off + 4 + bs > W.wave_end) {
      // the record is still open at the end of the wave: it becomes the next wave's carry
      if (!EMIT) {
        if (W.end_off <= W.wave_end) atomicAdd(&st->wave_chain, 1u);  // it would straddle the shard's end
        else if (W.final_wave) atomicAdd(&st->wave_trunc, 1u);
        else claim_carry(st, off, t ? (W.blocks[t - 1].coff << 16) | (off - lo) : st->carry_voff, t != 0);
      }
      open = true;
      break;
    }
    if (EMIT) {
      if (w + n < W.rec_cap) W.rec[w + n] = off | ((uint64_t)t << 40);
    } else {
      // l_seq is not validated yet (the facet kernel does that): only a length the record can hold counts
      uint32_t lseq = ld_u32_unaligned(W.d + off + 20);
      if ((uint64_t)lseq + (lseq + 1ull) / 2 + 32 <= bs) max_lseq = lseq > max_lseq ? lseq : max_lseq;
      else atomicAdd(&st->wave_bad, 1u);
    }
    ++n;
    off += 4 + bs;
  }
  if (EMIT) return;
  W.count[t] = n;
  if (max_lseq) atomicMax(&st->max_lseq, max_lseq);
  if (open) return;
  // closure: the walk must end on the shard's end, on the end of the wave, or on the first record of the block it lands in
  if (off >= W.end_off) {
    if (off != W.end_off) atomicAdd(&st->wave_chain, 1u);
    else st->wave_end_reached = 1;
    return;
  }
  if (off == W.wave_end) { claim_carry(st, off, 0, false); return; }
  uint32_t j = t;  // candidate landing block (t - 1 is this walk's own block; the carried record starts before block 0)
  while (j < W.n_blocks && block_lo(W, j) + W.blocks[j].isize <= off) {
    if (W.first[j] != kNoFirst) atomicAdd(&st->wave_chain, 1u);  // a record start claimed inside a record
    ++j;
  }
  if (j >= W.n_blocks) { atomicAdd(&st->wave_chain, 1u); return; }
  const uint64_t jlo = block_lo(W, j);
  if (W.first[j] == kNoFirst && off + 36 > W.wave_end && !W.final_wave && W.end_off > W.wave_end) {
    // too close to the end of the wave for find_first to judge it (no complete header): this is the carry
    claim_carry(st, off, (W.blocks[j].coff << 16) | (off - jlo), true);
    return;
  }
  if (W.first[j] == kNoFirst || jlo + W.first[j] != off) atomicAdd(&st->wave_chain, 1u);
  else W.landed[j] = 1;
}

// Every block that claims a first record (other than the root block) must have been landed on.
template <bool REDO>
__global__ void check_landed_kernel(WaveParams W) {
  const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= W.n_blocks) return;
  RunState* st = W.st;
  if (REDO && !st->redo) return;
  if (wave_dead(st)) return;
  if (W.first[b] == kNoFirst || W.landed[b]) return;
  const uint64_t root = wave_root(W);
  const uint64_t lo = block_lo(W, b);
  if (root >= lo && root < lo + W.blocks[b].isize) return;  // the root block starts the chain
  atomicAdd(&st->wave_chain, 1u);
}

// Serial fallback (one CTA): when closure failed, one thread walks the wave's chain from its root and fills first[]
// from scratch; the closure pass then runs again over the rebuilt table.
__global__ void __launch_bounds__(1024) chain_fix_kernel(WaveParams W) {
  RunState* st = W.st;
  if (wave_dead(st) || !st->wave_chain) return;
  for (uint32_t i = threadIdx.x; i < W.n_blocks; i += blockDim.x) { W.first[i] = kNoFirst; W.landed[i] = 0; }
  __syncthreads();
  if (threadIdx.x) return;
  st->wave_chain = st->wave_bad = st->wave_trunc = st->wave_end_reached = 0;
  st->next_carry = kNoCarry;
  st->redo = 1;
  const uint64_t d_end = W.end_off < W.wave_end ? W.end_off : W.wave_end;
  uint64_t off = wave_root(W);
  uint32_t b = 0;
  while (off < d_end) {
    if (off >= W.headroom) {
      while (b < W.n_blocks && block_lo(W, b) + W.blocks[b].isize <= off) ++b;
      if (b >= W.n_blocks) return;
      if (W.first[b] == kNoFirst) W.first[b] = (uint32_t)(off - block_lo(W, b));
    }
    if (off + 36 > W.wave_end) return;  // open at the end of the wave: the walk reports it
    uint32_t bs = ld_u32_unaligned(W.d + off);
    if (bs < 32 || bs > kMaxRecordBytes || off + 4 + bs > W.wave_end) return;
    off += 4 + bs;
  }
}

// Exclusive scan of the per-walk counts into table bases (single CTA, grid-stride over chunks), then the wave's
// commit: record count, next carry, errors.
__global__ void __launch_bounds__(1024) scan_counts_kernel(WaveParams W) {
  __shared__ uint64_t warp_sums[32];
  __shared__ uint64_t carry_s;
  RunState* st = W.st;
  const uint32_t n = W.n_blocks + 1;
  if (threadIdx.x == 0) carry_s = 0;
  __syncthreads();
  const uint32_t lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const bool live = !wave_dead(st);
  for (uint32_t start = 0; live && start < n; start += blockDim.x) {
    uint32_t i = start + threadIdx.x;
    uint64_t v = i < n ? W.count[i] : 0, x = v;
    for (int o = 1; o < 32; o <<= 1) {
      uint64_t y = __shfl_up_sync(0xFFFFFFFFu, x, o);
      if ((int)lane >= o) x += y;
    }
    if (lane == 31) warp_sums[wid] = x;
    __syncthreads();
    if (wid == 0) {
      uint64_t s = lane < (blockDim.x >> 5) ? warp_sums[lane] : 0;
      for (int o = 1; o < 32; o <<= 1) {
        uint64_t y = __shfl_up_sync(0xFFFFFFFFu, s, o);
        if ((int)lane >= o) s += y;
      }
      warp_sums[lane] = s;
    }
    __syncthreads();
    uint64_t carry = carry_s;
    uint64_t wbase = wid ? warp_sums[wid - 1] : 0;
    if (i < n) W.base[i] = carry + wbase + x - v;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry_s = carry + wbase + x;
    __syncthreads();
  }
  if (threadIdx.x) return;
  if (!live) { st->wave_rec = 0; return; }
  uint32_t fatal = 0;
  if (st->wave_chain) fatal |= kFatalChain;
  if (st->wave_trunc) fatal |= kFatalTruncated;
  if (st->wave_bad) fatal |= kFatalBadRecord;
  const uint64_t total = carry_s;
  if (total > W.rec_cap) fatal |= kFatalRecTable;
  if (st->wave_end_reached) {
    st->end_pending = 1;  // later waves hold nothing this shard owns (this wave's emit pass and facet kernels still run)
    st->cn_len = 0;
  } else if (st->next_carry == kNoCarry) {
    // nobody reached the end of the wave: only legal when the wave holds nothing of ours at all
    if (total || st->carry_len) fatal |= kFatalChain;
    st->cn_len = 0;
  } else {
    const uint64_t len = W.wave_end - st->next_carry;
    if (len > W.headroom) fatal |= kFatalCarry;
    st->cn_len = fatal ? 0u : (uint32_t)len;
    st->cn_src = st->next_carry;
    st->cn_voff = st->next_carry >= W.headroom ? st->next_carry_voff : st->carry_voff;  // below the headroom: the same record stays carried
  }
  st->wave_rec = fatal ? 0 : total;
  if (fatal) atomicOr(&st->fatal, fatal);
}

}  // namespace ngsq
