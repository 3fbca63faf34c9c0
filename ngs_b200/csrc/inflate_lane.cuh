// K2a — per-lane DEFLATE symbol decoder: ONE BGZF block per lane, 32 blocks per warp instruction
// (reference: the inflate noodles-bgzf/miniz_oxide perform under bam::Reader,
// src/utils/formats/bam.rs:41-44; format = RFC 1951 inside the BGZF framing of SAM spec 4.1).
//
// Huffman decoding never looks at the LZ77 window, so it is separated from the match copies:
//   * this decoder writes literals to their final positions (gathered into aligned 16-byte
//     chunks) and, for every match, a 3-byte token IN PLACE at the match destination
//     ((len-3) | (dist-1) << 8) plus one bit in a per-block bitmap (bit = match starts here);
//   * the warp-per-block resolve kernel (inflate2.cuh) then walks the bitmap in stream order and
//     performs the copies.
//
// Decoding is CANONICAL and branch-free, not table-driven: the code length of the next symbol is
// 1 + the number of per-length limits (left-aligned end of each length's code range, 16 x u16
// packed in 8 registers) that the next 15 bits reach, counted with packed 16-bit subtractions; the
// symbol is sorted[code + base[len]].  Every lane executes the same instructions whatever its code
// length (with a LUT + slow path a warp pays for both on nearly every symbol: ncu, profiles/), and
// the per-lane shared-memory footprint is 0.6 KB instead of 1.2-1.7 KB — shared memory is what
// bounds the number of resident decoders per SM.
//
// Everything in this file is scalar per-lane code with no warp intrinsics, so the same source
// also compiles for the host: tools/inflate_model.cpp runs it against zlib as a CPU model of the
// kernel (test tooling only; the product has no CPU path).
//
// Per-lane shared-memory slab (kSlabBytes, odd number of words so that equal indices of
// neighbouring lanes fall into different banks):
//   SL_LLBT  u32 ll_bt[15]       per code length: (index of first symbol - first code) & 0xFFFF
//                                | (index of the first symbol >= 256 of that length) << 16
//   SL_LLS   u8  ll_sorted[288]  literal/length symbols (& 255) in canonical order
//                                (while a dynamic header is parsed: the code-length-code LUT)
//   SL_DB    u8  d_base[15]      per code length: (index of first symbol - first code) mod 32
//   SL_DS    u8  d_sorted[32]    distance symbols in canonical order
// The 4-bit code lengths of a dynamic header and the build counters live in per-thread local
// memory (header() only; lanes of a warp parse their headers in lock step, so those accesses
// coalesce): shared memory is spent on what the symbol loop reads.
#pragma once
#include <stdint.h>
#include <string.h>

#if defined(__CUDACC__)
#define NGSQ_HD __host__ __device__ __forceinline__
#define NGSQ_HD_NOINLINE __host__ __device__ __noinline__
#else
#define NGSQ_HD inline
#define NGSQ_HD_NOINLINE
#endif

namespace ngsq {

// The symbol loop takes its length / distance bases from a 64-word table, stores under predicates instead of branching,
// and uses the 396-byte slab, which fits 18 decoder warps per SM instead of 17: the fastest of the forms measured on a
// B200 (profiles/round2_ab_inflate_variants.md: 36.6 -> 32.1 ms per 30 M records).

// ll_bt[15] and d_base[15] are indexed by length - 1 (length 16 = invalid code reads the neighbouring bytes of the
// slab; the block is failed anyway), distance bases are kept mod 32 in bytes: 60 + 288 + 15 + 32 = 395 -> 99 words
constexpr int SL_LLBT = 0, SL_LLS = 60, SL_DB = 348, SL_DS = 363;
constexpr int kSlabBytes = 396;
constexpr uint32_t kBitmapWords = 2048;  // per BGZF block: one bit per inflated byte (<= 65536)

enum : uint32_t { kBlkOk = 0, kBlkBadStream = 1, kBlkIsize = 2, kBlkOverrun = 3 };
enum : int { LS_HEADER = 0, LS_DECODE = 1, LS_IDLE = 2 };

struct BlockDesc {
  uint64_t in_off;   // absolute device address of the DEFLATE payload
  uint64_t out_off;  // offset of this block's first inflated byte in its wave (relative to the `out` the kernels get)
  uint32_t clen;     // DEFLATE payload length
  uint32_t isize;    // expected inflated size
  uint64_t coff;     // file offset of the BGZF block (virtual offsets of its records)
};

NGSQ_HD uint32_t brev32(uint32_t x) {
#if defined(__CUDA_ARCH__)
  return __brev(x);
#else
  x = ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
  x = ((x >> 2) & 0x33333333u) | ((x & 0x33333333u) << 2);
  x = ((x >> 4) & 0x0F0F0F0Fu) | ((x & 0x0F0F0F0Fu) << 4);
  x = ((x >> 8) & 0x00FF00FFu) | ((x & 0x00FF00FFu) << 8);
  return (x >> 16) | (x << 16);
#endif
}

// entry i < 32: length symbol 257 + i -> (match length - 3 base) | extra bits << 8;
// entry 32 + i: distance symbol i -> (distance - 1 base) | extra bits << 16
NGSQ_HD uint32_t base_lut_entry(uint32_t i) {
  if (i < 32) {
    const uint32_t li = i > 28 ? 28 : i;
    const uint32_t eb = (li < 8 || li == 28) ? 0 : (li - 4) >> 2;
    const uint32_t b = li < 8 ? li : li == 28 ? 255 : (4 + (li & 3)) << eb;
    return b | (eb << 8);
  }
  const uint32_t ds = (i - 32) > 29 ? 29 : (i - 32);
  const uint32_t deb = ds < 4 ? 0 : (ds >> 1) - 1;
  const uint32_t b = ds < 4 ? ds : (2 + (ds & 1)) << deb;
  return b | (deb << 16);
}

struct Quad { uint32_t x, y, z, w; };

NGSQ_HD Quad ld_in128(const uint8_t* p) {  // p is 16-byte aligned
  Quad q;
#if defined(__CUDA_ARCH__)
  uint4 v = __ldg(reinterpret_cast<const uint4*>(p));
  q.x = v.x; q.y = v.y; q.z = v.z; q.w = v.w;
#else
  memcpy(&q, p, 16);
#endif
  return q;
}

struct InflateCounters {  // host model only
  uint64_t symbols = 0, literals = 0, matches = 0, match_bytes = 0, headers = 0, stored = 0, fixed = 0, chunk_stores = 0,
           edge_stores = 0, ll_len_hist[17] = {0}, d_len_hist[17] = {0};
};

struct Lane {
  // bit reader: a 128-bit window {w0..w3} of the stream plus the next 64 bits {s0, s1} already
  // loaded; `pos` (< 64 after refill()) is the bit offset of the next unread bit in the window.
  // refill() slides the window by 64 bits when pos has passed 64 (the load it issues then is not
  // consumed before the next slide, >= 64 bits of symbols later) and snapshots the 64 bits at pos
  // into bb: one refill per symbol covers the worst case (48 bits: length + distance codes and
  // their extra bits).  ncu drove this shape: a word-at-a-time refill with two call sites cost a
  // quarter of the kernel's instructions.
  uint64_t bb;
  uint32_t w0, w1, w2, w3, s0, s1;
  uint32_t t0, t1;          // target of the load in flight; becomes {s0, s1} in settle()
  uint32_t shifted;         // a load into {t0, t1} has been issued and not settled yet
  uint32_t pos;
  const uint8_t* ptr;       // next 8 bytes to load (window base + 24)
  const uint8_t* in_end;
  // output, in "aligned coordinates": q = block-relative position + (address of the block & 15)
  uint8_t* obase;           // 16-byte aligned address of coordinate 0
  uint32_t q, q0, qend;
  uint64_t acc_lo, acc_hi;  // bytes of the current 16-byte chunk decided so far
  // match bitmap of this block
  uint32_t* bitmap;
  uint32_t bm, bm_w;
  // canonical-code limits: llim[i] = lim[2i] | lim[2i+1] << 16, lim[0] = 0x8000 (never reached)
  uint32_t llim[8], dlim[8];
  uint8_t* slab;            // shared memory (host model: heap)
  const uint32_t* lut;      // base_lut_entry(0..63)
  uint32_t err;
  int state;
  bool bfinal;
#ifdef NGSQ_HOST_MODEL
  InflateCounters* ctr;
#endif

  NGSQ_HD uint8_t* ll_sorted() const { return slab + SL_LLS; }
  NGSQ_HD uint32_t* ll_bt() const { return reinterpret_cast<uint32_t*>(slab + SL_LLBT) - 1; }  // index: code length
  NGSQ_HD uint8_t* d_sorted() const { return slab + SL_DS; }
  NGSQ_HD uint8_t* d_base() const { return slab + SL_DB - 1; }  // index: code length

  // ---------------- bit reader ----------------
  static NGSQ_HD void ld64(const uint8_t* p, uint32_t& lo, uint32_t& hi) {  // p is 8-byte aligned
#if defined(__CUDA_ARCH__)
    const uint2 v = __ldg(reinterpret_cast<const uint2*>(p));
    lo = v.x;
    hi = v.y;
#else
    memcpy(&lo, p, 4);
    memcpy(&hi, p + 4, 4);
#endif
  }
  static NGSQ_HD uint32_t funnel_r(uint32_t lo, uint32_t hi, uint32_t sh) {  // bits [sh, sh+32) of hi:lo, sh < 32
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, sh);
#else
    return sh ? (lo >> sh) | (hi << (32 - sh)) : lo;
#endif
  }
  NGSQ_HD void br_init(const uint8_t* p) {
    const uint32_t mis = (uint32_t)(reinterpret_cast<uintptr_t>(p) & 7);
    const uint8_t* base = p - mis;
    ld64(base, w0, w1);
    ld64(base + 8, w2, w3);
    ld64(base + 16, s0, s1);
    ptr = base + 24;
    pos = 8 * mis;
    shifted = 0;
    refill();
  }
  // The load issued by a slide goes to {t0, t1} and is copied to {s0, s1} by settle(), which the
  // symbol loop calls at the END of the iteration (a different basic block, a few hundred
  // instructions later).  Loading straight into {s0, s1} makes ptxas hoist the load above the
  // reads of s0/s1, park it in temporaries and copy them at once — a copy that waits for the load.
  NGSQ_HD void settle() {
    if (shifted) { s0 = t0; s1 = t1; shifted = 0; }
  }
  NGSQ_HD void refill() {
    if (pos >= 64) {
      w0 = w2; w1 = w3; w2 = s0; w3 = s1;
      ld64(ptr, t0, t1);
      ptr += 8;
      pos -= 64;
      shifted = 1;
    }
    const bool up = pos & 32;
    const uint32_t a = up ? w1 : w0, b = up ? w2 : w1, c = up ? w3 : w2;
    const uint32_t sh = pos & 31;
    bb = (uint64_t)funnel_r(a, b, sh) | ((uint64_t)funnel_r(b, c, sh) << 32);
  }
  NGSQ_HD void refill_cold() { refill(); settle(); }  // headers: latency does not matter
  NGSQ_HD uint32_t peek() const { return (uint32_t)bb; }
  NGSQ_HD void drop(uint32_t n) { bb >>= n; pos += n; }
  NGSQ_HD uint32_t take(uint32_t n) {
    uint32_t v = (uint32_t)bb & ((1u << n) - 1u);
    drop(n);
    return v;
  }
  // address of the next unread byte once the reader is byte-aligned
  NGSQ_HD const uint8_t* byte_ptr() const { return ptr - 24 + (pos >> 3); }
  // a malformed stream must not run away over the input: a valid one never reads past in_end
  NGSQ_HD bool overran() const { return byte_ptr() > in_end + 8; }

  // ---------------- output ----------------
  // Decided bytes are gathered into an aligned 16-byte chunk {acc_lo, acc_hi} and stored with one
  // 128-bit store; bytes of the chunk that belong to a match are stored as zero and overwritten by
  // the resolve kernel afterwards.  (Measured alternative: a 32-bit word accumulator needs 7 % fewer
  // instructions but its partial-sector stores raise the kernel's DRAM traffic from 1.3x to 1.6x of
  // C + D; the run time is the same.)
  NGSQ_HD void flush_chunk(uint32_t cq) {  // cq: multiple of 16; the chunk covers coordinates [cq, cq+16)
    if (cq >= q0 && cq + 16 <= qend) {
#if defined(__CUDA_ARCH__)
      *reinterpret_cast<uint4*>(obase + cq) = make_uint4((uint32_t)acc_lo, (uint32_t)(acc_lo >> 32), (uint32_t)acc_hi, (uint32_t)(acc_hi >> 32));
#else
      memcpy(obase + cq, &acc_lo, 8);
      memcpy(obase + cq + 8, &acc_hi, 8);
#endif
#ifdef NGSQ_HOST_MODEL
      if (ctr) ctr->chunk_stores++;
#endif
    } else {
      flush_edge(obase, q0, qend, acc_lo, acc_hi, cq);
#ifdef NGSQ_HOST_MODEL
      if (ctr) ctr->edge_stores++;
#endif
    }
  }
  // first / last chunk of the block shares its 16 bytes with the neighbouring block: bytes only
  // (static and by value: a non-inlined member call would force the whole Lane into local memory)
  static NGSQ_HD_NOINLINE void flush_edge(uint8_t* obase, uint32_t q0, uint32_t qend, uint64_t lo, uint64_t hi, uint32_t cq) {
#pragma unroll 1
    for (uint32_t i = 0; i < 16; ++i) {
      uint32_t c = cq + i;
      if (c >= q0 && c < qend) obase[c] = (uint8_t)((i < 8 ? lo >> (8 * i) : hi >> (8 * (i - 8))));
    }
  }
  // append the low n (1..3) bytes of v, then leave `sk` bytes to the resolve kernel
  NGSQ_HD void emit(uint32_t v, uint32_t n, uint32_t sk) {
    const uint32_t pos = q & 15;
    const uint32_t s = pos * 8;
    // 128-bit left shift of a 24-bit value by s in [0, 120], without shift counts >= 64
    const uint64_t V = v;
    const bool in_lo = s < 64;
    const uint32_t s6 = s & 63;
    const uint64_t up = V << s6;                 // s < 64: low half;  s >= 64: high half
    const uint64_t carry = (V >> 1) >> (63 - s6);  // s < 64: bits that cross into the high half
    acc_lo |= in_lo ? up : 0;
    acc_hi |= in_lo ? carry : up;
    const uint32_t nq = q + n;
    if ((nq ^ q) & 16) {  // chunk complete (possibly with bytes spilling into the next one)
      flush_chunk(q & ~15u);
      acc_lo = (pos + n > 16) ? (uint64_t)(v >> (8 * (16 - pos))) : 0;
      acc_hi = 0;
    }
    q = nq;
    if (sk) {
      const uint32_t sq = q + sk;
      if ((sq >> 4) != (q >> 4)) {
        if (q & 15) flush_chunk(q & ~15u);
        acc_lo = 0;
        acc_hi = 0;
      }
      q = sq;
    }
  }
  // stores under a predicate instead of a branch (device: one @p ST; host: an if)
  static NGSQ_HD void store16_if(bool c, uint8_t* p, uint64_t lo, uint64_t hi) {
#if defined(__CUDA_ARCH__)
    asm volatile("{\n\t.reg .pred p;\n\t.reg .u64 a;\n\tsetp.ne.u32 p, %0, 0;\n\tcvta.to.global.u64 a, %1;\n\t@p st.global.v4.u32 [a], {%2, %3, %4, %5};\n\t}"
                 :: "r"((uint32_t)c), "l"(p), "r"((uint32_t)lo), "r"((uint32_t)(lo >> 32)), "r"((uint32_t)hi), "r"((uint32_t)(hi >> 32)) : "memory");
#else
    if (c) { memcpy(p, &lo, 8); memcpy(p + 8, &hi, 8); }
#endif
  }
  static NGSQ_HD void store4_if(bool c, uint32_t* p, uint32_t v) {
#if defined(__CUDA_ARCH__)
    asm volatile("{\n\t.reg .pred p;\n\t.reg .u64 a;\n\tsetp.ne.u32 p, %0, 0;\n\tcvta.to.global.u64 a, %1;\n\t@p st.global.u32 [a], %2;\n\t}" :: "r"((uint32_t)c), "l"(p), "r"(v) : "memory");
#else
    if (c) *p = v;
#endif
  }
  NGSQ_HD void flush_chunk_if(bool c, uint32_t cq) {
    const bool inner = cq >= q0 && cq + 16 <= qend;
    store16_if(c && inner, obase + cq, acc_lo, acc_hi);
    if (c && !inner) flush_edge(obase, q0, qend, acc_lo, acc_hi, cq);  // first / last chunk of the block only
#ifdef NGSQ_HOST_MODEL
    if (ctr && c) { if (inner) ctr->chunk_stores++; else ctr->edge_stores++; }
#endif
  }
  NGSQ_HD void emit_sel(uint32_t v, uint32_t n, uint32_t sk) {  // same contract as emit()
    const uint32_t pos = q & 15;
    const uint32_t s = pos * 8;
    const uint64_t V = v;
    const bool in_lo = s < 64;
    const uint32_t s6 = s & 63;
    const uint64_t up = V << s6;
    const uint64_t carry = (V >> 1) >> (63 - s6);
    acc_lo |= in_lo ? up : 0;
    acc_hi |= in_lo ? carry : up;
    const uint32_t nq = q + n;
    const bool cross1 = ((nq ^ q) & 16) != 0;  // the token completes this chunk
    flush_chunk_if(cross1, q & ~15u);
    // bytes of the token that spill into the next chunk: 16 - pos is 1..3 whenever cross1 holds (n <= 3),
    // and the shifted-out value is 0 when the token ends exactly at the boundary
    const uint32_t left = v >> ((8 * (16 - pos)) & 31);
    acc_lo = cross1 ? (uint64_t)left : acc_lo;
    acc_hi = cross1 ? 0 : acc_hi;
    const uint32_t sq = nq + sk;
    const bool cross2 = (sq >> 4) != (nq >> 4);  // the match bytes left to the resolve kernel leave the chunk
    flush_chunk_if(cross2 && (nq & 15), nq & ~15u);
    acc_lo = cross2 ? 0 : acc_lo;
    acc_hi = cross2 ? 0 : acc_hi;
    q = sq;
  }
  NGSQ_HD void mark_match_if(bool ok, uint32_t p) {
    const uint32_t w = p >> 5;
    const bool nw = ok && w != bm_w;
    store4_if(nw && bm != 0, bitmap + bm_w, bm);
    bm = nw ? 0 : bm;
    bm_w = nw ? w : bm_w;
    bm |= ok ? 1u << (p & 31) : 0u;
  }
  NGSQ_HD void finish_output() {
    if (q & 15) flush_chunk(q & ~15u);
    acc_lo = 0;
    acc_hi = 0;
    if (bm) bitmap[bm_w] = bm;
    bm = 0;
  }

  NGSQ_HD void begin_block(const BlockDesc& d, uint8_t* out, uint32_t* bitmap_of_block) {
    uint8_t* o = out + d.out_off;
    uint32_t ab = (uint32_t)(reinterpret_cast<uintptr_t>(o) & 15);
    obase = o - ab;
    q0 = ab;
    q = ab;
    qend = ab + d.isize;
    acc_lo = 0;
    acc_hi = 0;
    bitmap = bitmap_of_block;
    bm = 0;
    bm_w = 0;
    err = 0;
    bfinal = false;
    in_end = reinterpret_cast<const uint8_t*>(d.in_off) + d.clen;
    br_init(reinterpret_cast<const uint8_t*>(d.in_off));
    state = LS_HEADER;
  }
  NGSQ_HD void end_block(uint32_t e) {
    if (!e && q != qend) e = kBlkIsize;
    err = e;
    finish_output();
    state = LS_IDLE;
  }

  // ---------------- canonical tables ----------------
  // lens(k): code length of symbol k in [0, n).  Fills sorted[], the per-length bases and the
  // packed limits.  Literal/length table: bt32 != nullptr and `split` = 256 (the index of the first
  // symbol >= split of each length goes into the high half of bt32[]); distance table: base8.
  template <class LenFn>
  NGSQ_HD bool build(LenFn lens, uint32_t n, uint8_t* sorted, uint32_t* lim_packed, uint32_t* bt32, uint8_t* base8, uint32_t split,
                     uint16_t* nx /* scratch[16] */) {
    for (int i = 0; i < 16; ++i) nx[i] = 0;
    for (uint32_t k = 0; k < n; ++k) nx[lens(k)]++;
    nx[0] = 0;
    int left = 1;
    uint32_t code = 0, off = 0, prev = 0, lim_lo = 0x8000u;
#pragma unroll
    for (int l = 1; l <= 15; ++l) {  // unrolled: lim_packed[] lives in registers (static indices only)
      const uint32_t c = nx[l];
      left = (left << 1) - (int)c;
      if (left < 0) return false;  // over-subscribed
      code = (code + prev) << 1;
      prev = c;
      const uint32_t lim = (code + c) << (15 - l);  // <= 0x8000
      if (l & 1) lim_packed[l >> 1] = lim_lo | (lim << 16); else lim_lo = lim;
      const int b = (int)off - (int)code;
      if (bt32) bt32[l] = ((uint32_t)b & 0xFFFFu) | (off << 16); else base8[l] = (uint8_t)b;  // used mod 32
      nx[l] = (uint16_t)off;  // running index of the next symbol of this length
      off += c;
    }
    if (left > 0 && off > 1) return false;  // incomplete with two or more codes (zero or one used symbol is accepted)
    for (uint32_t k = 0; k < n; ++k) {
      const uint32_t l = lens(k);
      if (!l) continue;
      const uint32_t i = nx[l];
      nx[l] = (uint16_t)(i + 1);
      sorted[i] = (uint8_t)k;
      if (bt32 && k < split) bt32[l] += 1u << 16;  // literals come first within a length: count them
    }
    return true;
  }

  // code length of the next symbol: 1 + number of limits the next 15 bits (MSB first) reach
  static NGSQ_HD uint32_t code_len(uint32_t x, const uint32_t* lim_packed) {
    const uint32_t x2 = (x * 0x10001u) | 0x80008000u;
#if defined(__CUDA_ARCH__)
    // bit 15 of each half of (x2 - lim) says x >= lim: gather the 16 flag bytes with four byte
    // permutes, interleave their top bits into one word, popcount
    const uint32_t g0 = __byte_perm(x2 - lim_packed[0], x2 - lim_packed[1], 0x7531);
    const uint32_t g1 = __byte_perm(x2 - lim_packed[2], x2 - lim_packed[3], 0x7531);
    const uint32_t g2 = __byte_perm(x2 - lim_packed[4], x2 - lim_packed[5], 0x7531);
    const uint32_t g3 = __byte_perm(x2 - lim_packed[6], x2 - lim_packed[7], 0x7531);
    uint32_t r = g3 & 0x80808080u;
    r = (g2 & 0x80808080u) | (r >> 1);
    r = (g1 & 0x80808080u) | (r >> 1);
    r = (g0 & 0x80808080u) | (r >> 1);
    return __popc(r) + 1;
#else
    uint32_t s = 0;
    for (int i = 0; i < 8; ++i) s += ((x2 - lim_packed[i]) >> 15) & 0x10001u;
    return (s & 0xFFFFu) + (s >> 16) + 1;
#endif
  }

  // ---------------- DEFLATE block header (+ stored blocks) ----------------
  NGSQ_HD void header() {
    refill_cold();
    uint32_t h = take(3);
    bfinal = h & 1;
    uint32_t btype = h >> 1;
#ifdef NGSQ_HOST_MODEL
    if (ctr) ctr->headers++;
#endif
    if (btype == 3) { end_block(kBlkBadStream); return; }
    if (btype == 0) {
#ifdef NGSQ_HOST_MODEL
      if (ctr) ctr->stored++;
#endif
      drop((0u - pos) & 7u);  // to the next byte boundary
      refill_cold();
      uint32_t v = take(16);
      refill_cold();
      uint32_t nv = take(16);
      if ((v ^ nv) != 0xFFFFu) { end_block(kBlkBadStream); return; }
      const uint8_t* sp = byte_ptr();
      if (q + v > qend || sp + v > in_end) { end_block(kBlkOverrun); return; }
      for (uint32_t k = 0; k < v; ++k) emit(sp[k], 1, 0);
      br_init(sp + v);
      if (bfinal) end_block(0);
      return;  // state stays LS_HEADER otherwise
    }
    bool ok;
    uint16_t scratch[16];
    if (btype == 1) {
#ifdef NGSQ_HOST_MODEL
      if (ctr) ctr->fixed++;
#endif
      ok = build([](uint32_t k) -> uint32_t { return k < 144 ? 8u : k < 256 ? 9u : k < 280 ? 7u : 8u; }, 288, ll_sorted(), llim, ll_bt(), nullptr, 256, scratch);
      ok = ok && build([](uint32_t) -> uint32_t { return 5u; }, 32, d_sorted(), dlim, nullptr, d_base(), 0, scratch);
    } else {
      refill_cold();
      uint32_t v = take(14);
      const uint32_t hlit = (v & 31) + 257, hdist = ((v >> 5) & 31) + 1, hclen = ((v >> 10) & 15) + 4;
      if (hlit > 286 || hdist > 30) { end_block(kBlkBadStream); return; }
      // 19 code-length-code lengths, 3 bits each, kept in one register
      uint64_t clpack = 0;
      for (uint32_t i = 0; i < hclen; ++i) {
        refill_cold();
        // order: 16 17 18 0 8 7 9 6 10 5 11 4 12 3 13 2 14 1 15
        const uint64_t order = 0xF1E2D3C4B5A69780ull;  // nibbles for i = 3..18
        uint32_t sym = i < 3 ? 16 + i : (uint32_t)((order >> (4 * (i - 3))) & 15);
        clpack |= (uint64_t)take(3) << (3 * sym);
      }
      // code-length code: canonical, 7-bit LUT (aliases ll_sorted): (sym << 3) | len
      uint8_t* cl_lut = slab + SL_LLS;
      {
        uint32_t c[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int k = 0; k < 19; ++k) {
          uint32_t l = (uint32_t)(clpack >> (3 * k)) & 7;
#pragma unroll
          for (int t = 1; t < 8; ++t) c[t] += (l == (uint32_t)t);
        }
        uint32_t nx[8];
        uint32_t code = 0, prev = 0, used = 0;
        int left = 1;
        nx[0] = 0;
#pragma unroll
        for (int l = 1; l <= 7; ++l) {
          left = (left << 1) - (int)c[l];
          code = (code + prev) << 1;
          prev = c[l];
          nx[l] = code;
          used += c[l];
        }
        // over-subscribed, or incomplete with two or more codes
        if (left < 0 || (left > 0 && used > 1)) { end_block(kBlkBadStream); return; }
        uint32_t* lw = reinterpret_cast<uint32_t*>(cl_lut);
        for (int i = 0; i < 32; ++i) lw[i] = 0;
        for (int k = 0; k < 19; ++k) {
          uint32_t l = (uint32_t)(clpack >> (3 * k)) & 7;
          if (!l) continue;
          uint32_t cd = 0;
#pragma unroll
          for (int t = 1; t < 8; ++t)
            if (l == (uint32_t)t) { cd = nx[t]; nx[t] = cd + 1; }
          for (uint32_t j = brev32(cd) >> (32 - l); j < 128; j += (1u << l)) cl_lut[j] = (uint8_t)((k << 3) | l);
        }
      }
      // hlit + hdist code lengths as nibbles, eight per stored word
      uint32_t nb[40];
      const uint32_t* nbp = nb;
      const uint32_t total = hlit + hdist;
      uint32_t i = 0, word = 0, prevlen = 0;
      bool bad = false;
      while (i < total) {
        refill_cold();
        if (overran()) { bad = true; break; }
        uint32_t e = cl_lut[peek() & 127];
        uint32_t l = e & 7, sym = e >> 3;
        if (!l) { bad = true; break; }
        drop(l);
        uint32_t rep = 1, val = sym;
        if (sym == 16) { if (i == 0) { bad = true; break; } val = prevlen; rep = 3 + take(2); }
        else if (sym == 17) { val = 0; rep = 3 + take(3); }
        else if (sym == 18) { val = 0; rep = 11 + take(7); }
        if (i + rep > total) { bad = true; break; }
        prevlen = val;
        for (uint32_t k = 0; k < rep; ++k) {
          word |= val << (4 * (i & 7));
          ++i;
          if (!(i & 7)) { nb[(i >> 3) - 1] = word; word = 0; }
        }
      }
      if (i & 7) nb[i >> 3] = word;
      if (bad) { end_block(kBlkBadStream); return; }
      if (((nb[256 >> 3] >> (4 * (256 & 7))) & 15) == 0) { end_block(kBlkBadStream); return; }  // no end-of-block code
      ok = build([nbp](uint32_t k) -> uint32_t { return (nbp[k >> 3] >> (4 * (k & 7))) & 15; }, hlit, ll_sorted(), llim, ll_bt(), nullptr, 256, scratch);
      ok = ok && build([nbp, hlit](uint32_t k) -> uint32_t { const uint32_t j = hlit + k; return (nbp[j >> 3] >> (4 * (j & 7))) & 15; }, hdist,
                       d_sorted(), dlim, nullptr, d_base(), 0, scratch);
    }
    if (!ok) { end_block(kBlkBadStream); return; }
    state = LS_DECODE;
  }

  // ---------------- one literal/length(+distance) symbol ----------------
  // Straight-line on purpose: every warp step runs the union of the paths its lanes take and waits
  // out every branch (ncu: each warp is bound by its own dependency / branch-resolve latency, not by
  // issue slots), so range checks only accumulate flags that are tested once at the end, and the
  // length / distance bases are looked up without branches.  Out-of-range values are clamped where
  // they index memory; a flagged block is failed and never reaches the resolve kernel.
  NGSQ_HD void step() {
    refill();
    const uint32_t x = brev32(peek()) >> 17;
    const uint32_t len = code_len(x, llim);             // 1..15, 16 = bits beyond an incomplete code
    uint32_t bad_stream = len >> 4, overrun = 0;
    const uint32_t bt = ll_bt()[len];  // 1..16
    const uint32_t idx = ((x >> ((15 - len) & 31)) + bt) & 0xFFFFu;  // index into sorted (the base is kept mod 2^16)
    const uint32_t s8 = ll_sorted()[idx < 288 ? idx : 0];
    const bool upper = idx >= (bt >> 16);  // symbol >= 256
    drop(len);
#ifdef NGSQ_HOST_MODEL
    if (ctr) { ctr->symbols++; ctr->ll_len_hist[len]++; }
#endif
    uint32_t v = s8, n = 1, sk = 0;
    if (upper) {
      if (s8 == 0 && !bad_stream) {  // end of block
        if (overran()) { end_block(kBlkBadStream); return; }
        if (bfinal) end_block(0); else state = LS_HEADER;
        return;
      }
      // length symbol 257 + li: li < 8: 3 + li;  li = 28: 258;  else 3 + ((4 + (li & 3)) << eb) + extra, eb = (li - 4) >> 2
      const uint32_t li = s8 - 1;
      bad_stream |= li > 28;
      const uint32_t le = lut[li & 31];
      const uint32_t mlen = 3 + (le & 255) + take(le >> 8);
      const uint32_t dx = brev32(peek()) >> 17;
      const uint32_t dl = code_len(dx, dlim);
      bad_stream |= dl >> 4;
      const uint32_t di = ((dx >> ((15 - dl) & 31)) + (uint32_t)d_base()[dl]) & 31u;
      const uint32_t ds = d_sorted()[di];
      bad_stream |= ds > 29;
      drop(dl);
#ifdef NGSQ_HOST_MODEL
      if (ctr) ctr->d_len_hist[dl]++;
#endif
      // distance symbol ds: ds < 4: 1 + ds;  else 1 + ((2 + (ds & 1)) << deb) + extra, deb = (ds >> 1) - 1
      const uint32_t de = lut[32 + (ds & 31)];
      const uint32_t dist = 1 + (de & 0xFFFFu) + take(de >> 16);
      const uint32_t p = q - q0;
      overrun |= (dist > p) | (q + mlen > qend);
      mark_match_if(!(bad_stream | overrun), p);
      v = (mlen - 3) | ((dist - 1) << 8);
      n = 3;
      sk = mlen - 3;
#ifdef NGSQ_HOST_MODEL
      if (ctr) { ctr->matches++; ctr->match_bytes += mlen; }
#endif
    } else {
      overrun |= q >= qend;
#ifdef NGSQ_HOST_MODEL
      if (ctr) ctr->literals++;
#endif
    }
    if (bad_stream | overrun) { end_block(bad_stream ? kBlkBadStream : kBlkOverrun); return; }
    emit_sel(v, n, sk);
  }
};

}  // namespace ngsq
