// K2 — BGZF inflate as two kernels (reference: the inflate noodles-bgzf/miniz_oxide perform
// under bam::Reader, src/utils/formats/bam.rs:41-44, src/qc/command.rs:305 and :350).
//
//   inflate_decode_kernel   one BGZF block per LANE: 32 independent Huffman decoders per warp
//                           instruction (inflate_lane.cuh).  Literals go to their final place,
//                           matches leave a 3-byte token in place + a bit in the block's bitmap.
//                           Persistent grid, one CTA per SM (shared-memory bound: one table slab
//                           per lane); a warp pulls 32 consecutive blocks at a time so that the
//                           lanes of a warp meet their DEFLATE block headers together (zlib ends a
//                           block every 16383 symbols) and parse/build them in lock step.
//   inflate_resolve_kernel  one BGZF block per WARP: walks the bitmap in stream order, 32 tokens
//                           per step, one lane per LZ77 match; a match waits while its source
//                           still overlaps an unresolved earlier match.
// Both are issue/L1-bound integer kernels; HBM traffic is C + D (+ D/8 bitmap) per pass.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "inflate_lane.cuh"

namespace ngsq {

constexpr int kDecBatch = 32;  // symbols per lane between header / overrun checks
constexpr int kDecWarps = 18;  // 18 x 32 x 396 B of slabs + 256 B of static shared memory (s_base_lut)
constexpr int kDecThreads = kDecWarps * 32;
constexpr size_t kDecSmem = (size_t)kDecThreads * kSlabBytes;

__global__ void __launch_bounds__(kDecThreads, 1)
inflate_decode_kernel(uint8_t* __restrict__ out, const BlockDesc* __restrict__ blocks, uint32_t n_blocks,
                      uint32_t* __restrict__ queue, uint32_t* __restrict__ status, uint32_t* __restrict__ bitmap) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const uint32_t lane = threadIdx.x & 31;
  Lane L;
  L.slab = smem_raw + (size_t)threadIdx.x * kSlabBytes;
  L.state = LS_IDLE;
  __shared__ uint32_t s_base_lut[64];
  if (threadIdx.x < 64) s_base_lut[threadIdx.x] = base_lut_entry(threadIdx.x);
  __syncthreads();
  L.lut = s_base_lut;
  // First batch of every warp: static and interleaved over the CTAs (warp w of CTA c takes batch w * grid + c), so that a
  // partial wave — the tail of a run — spreads over all SMs with few warps each instead of filling a few SMs with 18: a
  // lane decodes its block serially, and a warp that shares its scheduler with four others runs at a fraction of the
  // speed of one that does not.  Later batches (launches larger than the grid) come from the queue.
  const uint32_t static_blocks = gridDim.x * (uint32_t)kDecWarps * 32u;
  bool first = true;
  for (;;) {
    uint32_t base = 0;
    if (first) {
      base = ((threadIdx.x >> 5) * gridDim.x + blockIdx.x) * 32u;
      first = false;
    } else {
      if (lane == 0) base = static_blocks + atomicAdd(queue, 32u);
      base = __shfl_sync(0xFFFFFFFFu, base, 0);
    }
    if (base >= n_blocks) break;
    const uint32_t b = base + lane;
    if (b < n_blocks) L.begin_block(blocks[b], out, bitmap + (size_t)b * kBitmapWords);
    else L.state = LS_IDLE;
    while (__any_sync(0xFFFFFFFFu, L.state != LS_IDLE)) {
      if (L.state == LS_HEADER) L.header();
      __syncwarp();
#pragma unroll 1
      for (int it = 0; it < kDecBatch; ++it) {
        if (L.state == LS_DECODE) L.step();
        L.settle();  // the input load of this iteration's window slide, consumed only here
        if (!__any_sync(0xFFFFFFFFu, L.state == LS_DECODE)) break;
      }
      if (L.state == LS_DECODE && L.overran()) L.end_block(kBlkBadStream);
    }
    if (b < n_blocks && L.err) status[b] = L.err;
  }
}

// The resolve kernel's dependency masks come from the bitmap's ranks (two popcounts over the super-window's bitmap words +
// one look at the preceding token): 2 shared-memory loads + 1 shuffle instead of the 12 shuffles of two binary searches
// over the lanes' destinations, which give the same masks (tools/inflate_model.cpp checks the equality on every batch).
// Measured on a B200, 30 M records: 29.3 -> 25.7 ms (profiles/round2_ab_inflate_variants.md).
constexpr int kResThreads = 256;
constexpr int kResWarps = kResThreads / 32;
constexpr int kResList = 352;  // matches that can start inside 1024 bytes (every match is >= 3 bytes)

// the 8 bytes at s (any alignment) through up to three aligned 32-bit loads and two funnel shifts: one
// L1 wavefront per lane per load instead of one per byte (the resolve kernel is L1-wavefront bound)
// (only the first n bytes are used: the third word is fetched only when they reach into it — most matches of BAM data are 3-5 bytes)
__device__ __forceinline__ uint2 load8_unaligned(const uint8_t* s, uint32_t n) {
  const uint32_t* a = reinterpret_cast<const uint32_t*>(reinterpret_cast<uintptr_t>(s) & ~uintptr_t(3));
  const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(s) & 3);
  const uint32_t sh = mis * 8;
  const uint32_t w0 = a[0], w1 = a[1];
  uint32_t w2 = 0;
  if (mis + n > 8) w2 = a[2];
  return make_uint2(__funnelshift_r(w0, w1, sh), __funnelshift_r(w1, w2, sh));
}

__device__ __forceinline__ void store_bytes(uint8_t* d, uint2 v, uint32_t n) {  // n in 1..8
  d[0] = (uint8_t)v.x;
  if (n > 1) d[1] = (uint8_t)(v.x >> 8);
  if (n > 2) d[2] = (uint8_t)(v.x >> 16);
  if (n > 3) d[3] = (uint8_t)(v.x >> 24);
  if (n > 4) d[4] = (uint8_t)v.y;
  if (n > 5) d[5] = (uint8_t)(v.y >> 8);
  if (n > 6) d[6] = (uint8_t)(v.y >> 16);
  if (n > 7) d[7] = (uint8_t)(v.y >> 24);
}

// One lane copies one match, 8 bytes per step.  A step copies from D bytes back, D a multiple of the
// match distance: D = dist while dist >= 8; for shorter periods D doubles after every step (the
// bytes written so far extend the periodic run), so overlapping runs need log2(8/dist) extra steps
// instead of a byte loop.  Every step reads only final bytes or bytes this lane wrote earlier.
__device__ __forceinline__ void resolve_copy(uint8_t* dst, uint32_t mlen, uint32_t dist) {
  uint32_t D = dist;
  for (uint32_t done = 0; done < mlen;) {
    const uint32_t n = min(min(8u, D), mlen - done);
    store_bytes(dst + done, load8_unaligned(dst + done - D, n), n);
    done += n;
    if (D < 8) D <<= 1;
  }
}

__global__ void __launch_bounds__(kResThreads)
inflate_resolve_kernel(uint8_t* __restrict__ out, const BlockDesc* __restrict__ blocks, uint32_t n_blocks,
                       const uint32_t* __restrict__ bitmap, const uint32_t* __restrict__ status) {
  __shared__ uint16_t s_pos[kResWarps][kResList];
  __shared__ uint2 s_rank[kResWarps][32];
  const uint32_t lane = threadIdx.x & 31, wic = threadIdx.x >> 5;
  const uint32_t n_warps = gridDim.x * kResWarps;
  uint16_t* list = s_pos[wic];
  for (uint32_t b = blockIdx.x * kResWarps + wic; b < n_blocks; b += n_warps) {
    if (status[b]) continue;  // failed blocks carry no trustworthy tokens
    const BlockDesc d = blocks[b];
    uint8_t* ob = out + d.out_off;
    const uint32_t* bmp = bitmap + (size_t)b * kBitmapWords;
    const uint32_t n_sw = (d.isize + 1023) >> 10;
    for (uint32_t sw = 0; sw < n_sw; ++sw) {
      uint32_t word = bmp[sw * 32 + lane];
      const uint32_t cnt = __popc(word);
      uint32_t incl = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, o);
        if ((int)lane >= o) incl += t;
      }
      const uint32_t total = __shfl_sync(0xFFFFFFFFu, incl, 31);
      if (!total) continue;
      uint32_t o = incl - cnt;
      // entry w: bitmap word w of this super-window and the number of matches that start before it (shared memory
      // rather than shuffles: the kernel runs at 32 registers per thread for full occupancy)
      s_rank[wic][lane] = make_uint2(word, o);
      const uint32_t pbase = (sw << 10) + (lane << 5);
      while (word) {
        const uint32_t bit = __ffs(word) - 1;
        word &= word - 1;
        list[o++] = (uint16_t)(pbase + bit);
      }
      __syncwarp();
      // token of the first batch; later batches are fetched one batch ahead (their bytes sit in
      // their own destinations, which no earlier copy touches)
      uint32_t pos_n = 0xFFFFu, tok_n = 0;
      if (lane < total) {
        pos_n = list[lane];
        const uint8_t* t = ob + pos_n;
        tok_n = (uint32_t)t[0] | ((uint32_t)t[1] << 8) | ((uint32_t)t[2] << 16);
      }
      for (uint32_t base = 0; base < total; base += 32) {
        const bool active = base + lane < total;
        const uint32_t pos = pos_n, tok = tok_n;
        const uint32_t jn = base + 32 + lane;
        if (jn < total) {
          pos_n = list[jn];
          const uint8_t* t = ob + pos_n;
          tok_n = (uint32_t)t[0] | ((uint32_t)t[1] << 8) | ((uint32_t)t[2] << 16);
        }
        const uint32_t mlen = (tok & 255u) + 3u, dist = (tok >> 8) + 1u;
        // destinations [pos, dend) are ascending and disjoint across lanes (inactive lanes: empty at the top)
        const uint32_t dend = active ? pos + mlen : 0x20000u;
        const uint32_t s_lo = pos - dist, s_hi = s_lo + min(mlen, dist);  // source bytes [s_lo, s_hi)
        // earlier lanes whose destination overlaps my source: lanes [lo, hi) with
        //   lo = first lane with dend > s_lo,  hi = first lane with pos >= s_hi
        // rank(x) = matches of this super-window that start before window-relative byte x: the matches that start inside
        // my source are the list entries [rank(s_lo), rank(s_hi)); the one before them counts if it reaches past s_lo.
        // Matches of earlier batches and earlier super-windows are resolved already.
        const uint32_t W = sw << 10;
        const uint32_t x_lo = min(max(s_lo, W) - W, 1023u), x_hi = min(max(s_hi, W) - W, 1023u);
        const uint2 e_lo = s_rank[wic][x_lo >> 5], e_hi = s_rank[wic][x_hi >> 5];
        const uint32_t r_lo = e_lo.y + __popc(e_lo.x & ((1u << (x_lo & 31)) - 1u));
        const uint32_t r_hi = e_hi.y + __popc(e_hi.x & ((1u << (x_hi & 31)) - 1u));
        const int pl = (int)r_lo - 1 - (int)base;  // lane of the match before my source, if it is in this batch
        const uint32_t prev_end = __shfl_sync(0xFFFFFFFFu, dend, pl & 31);
        const int lo = max((int)r_lo - (int)base - ((pl >= 0 && prev_end > s_lo) ? 1 : 0), 0), hi = (int)r_hi - (int)base;
        uint32_t dep = 0;
        if (active && hi > lo) dep = ((1u << hi) - 1u) & ~((1u << lo) - 1u) & ((1u << lane) - 1u);  // hi <= lane
        uint32_t done = __ballot_sync(0xFFFFFFFFu, !active);
        while (done != 0xFFFFFFFFu) {
          const bool ready = !((done >> lane) & 1u) && (dep & ~done) == 0;
          if (ready) resolve_copy(ob + pos, mlen, dist);
          __syncwarp();
          done |= __ballot_sync(0xFFFFFFFFu, ready);
        }
      }
      __syncwarp();
    }
  }
}

}  // namespace ngsq
