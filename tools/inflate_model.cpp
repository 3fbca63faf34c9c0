// CPU model of the v2 inflate kernels (test tooling; NOT part of the product library).
// Compiles ngs_b200/csrc/inflate_lane.cuh for the host, runs the per-lane decoder plus a scalar
// restatement of the resolve pass over every BGZF block of a file, checks the bytes against zlib
// and prints symbol statistics that drive kernel design decisions.
//   g++ -O2 -std=c++17 -DNGSQ_HOST_MODEL -o /tmp/inflate_model tools/inflate_model.cpp -lz
//   /tmp/inflate_model file.bam [max_blocks]
//   /tmp/inflate_model file.bam --fuzz N     N corrupted copies of every block: the decoder must fail
//                                            or finish, never write outside its block, never run away
//   /tmp/inflate_model file.bam --all-alignments   decode and resolve every block at all 16 output alignments
//                                            (the first with the scalar resolve pass, the others with the warp one)
//   /tmp/inflate_model file.bam --expect-reject    every block is invalid: the decoder must fail it (at every
//                                            output alignment), write nothing outside it, and zlib must reject it
#include <zlib.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <vector>

#include "../ngs_b200/csrc/inflate_lane.cuh"

using namespace ngsq;

// Lane-by-lane restatement of inflate_resolve_kernel (inflate2.cuh): 1024-byte super-windows, 32-token
// batches, dependency masks from two binary searches over the sorted destination ranges, rounds, and the
// 8-byte copy steps with distance doubling.  Reads of a round see memory as it was when the round
// started only where the kernel guarantees it (ready lanes never read what another ready lane writes).
static void resolve_copy_model(uint8_t* dst, uint32_t mlen, uint32_t dist) {
  uint32_t D = dist;
  for (uint32_t done = 0; done < mlen;) {
    const uint32_t n = std::min(std::min(8u, D), mlen - done);
    uint8_t tmp[8];
    memcpy(tmp, dst + done - D, n);  // the kernel loads the 8 bytes first, then stores n of them
    memcpy(dst + done, tmp, n);
    done += n;
    if (D < 8) D <<= 1;
  }
}

static uint64_t g_rounds = 0, g_batches = 0;

static void resolve_block_model(uint8_t* ob, uint32_t isize, const uint32_t* bitmap) {
  const uint32_t n_sw = (isize + 1023) >> 10;
  std::vector<uint32_t> list;
  for (uint32_t sw = 0; sw < n_sw; ++sw) {
    list.clear();
    for (uint32_t lane = 0; lane < 32; ++lane)
      for (uint32_t m = bitmap[sw * 32 + lane]; m; m &= m - 1) list.push_back((sw << 10) + (lane << 5) + __builtin_ctz(m));
    const uint32_t total = (uint32_t)list.size();
    for (uint32_t base = 0; base < total; base += 32) {
      uint32_t pos[32], mlen[32], dist[32], dpos[32], dend[32], s_lo[32], s_hi[32], dep[32];
      bool active[32];
      for (uint32_t l = 0; l < 32; ++l) {
        active[l] = base + l < total;
        pos[l] = active[l] ? list[base + l] : 0xFFFFu;
        uint32_t tok = 0;
        if (active[l]) tok = ob[pos[l]] | (ob[pos[l] + 1] << 8) | (ob[pos[l] + 2] << 16);  // tokens are read before any copy of the batch
        mlen[l] = (tok & 255u) + 3u;
        dist[l] = (tok >> 8) + 1u;
        dpos[l] = active[l] ? pos[l] : 0x20000u;
        dend[l] = active[l] ? pos[l] + mlen[l] : 0x20000u;
        s_lo[l] = pos[l] - dist[l];
        s_hi[l] = s_lo[l] + std::min(mlen[l], dist[l]);
      }
      for (uint32_t l = 0; l < 32; ++l) {
        uint32_t lo = 0, hi = 0;
        for (int step = 32; step; step >>= 1) {
          const uint32_t il = lo + step - 1, ih = hi + step - 1;
          const uint32_t e = dend[il & 31], p2 = dpos[ih & 31];
          if (il < 32 && e <= s_lo[l]) lo += step;
          if (ih < 32 && p2 < s_hi[l]) hi += step;
        }
        dep[l] = 0;
        if (active[l] && hi > lo) dep[l] = (hi >= 32 ? 0xFFFFFFFFu : ((1u << hi) - 1u)) & ~((1u << lo) - 1u) & ((1u << l) - 1u);
        // the rank masks of inflate2.cuh must give the same mask
        {
          const uint32_t W = sw << 10;
          const uint32_t x_lo = std::min(std::max(s_lo[l], W) - W, 1023u), x_hi = std::min(std::max(s_hi[l], W) - W, 1023u);
          auto rank = [&](uint32_t x) {
            uint32_t excl = 0;
            for (uint32_t w = 0; w < (x >> 5); ++w) excl += (uint32_t)__builtin_popcount(bitmap[sw * 32 + w]);
            return excl + (uint32_t)__builtin_popcount(bitmap[sw * 32 + (x >> 5)] & ((1u << (x & 31)) - 1u));
          };
          const uint32_t r_lo = rank(x_lo), r_hi = rank(x_hi);
          const int pl = (int)r_lo - 1 - (int)base;
          const uint32_t prev_end = dend[pl & 31];
          const int lo2 = std::max((int)r_lo - (int)base - ((pl >= 0 && prev_end > s_lo[l]) ? 1 : 0), 0), hi2 = (int)r_hi - (int)base;
          uint32_t dep2 = 0;
          if (active[l] && hi2 > lo2) dep2 = ((1u << hi2) - 1u) & ~((1u << lo2) - 1u) & ((1u << l) - 1u);
          if (dep2 != dep[l]) { fprintf(stderr, "resolve model: rank-based mask %08x != searched mask %08x (lane %u)\n", dep2, dep[l], l); exit(1); }
        }
      }
      uint32_t done = 0;
      for (uint32_t l = 0; l < 32; ++l) if (!active[l]) done |= 1u << l;
      g_batches++;
      while (done != 0xFFFFFFFFu) {
        uint32_t ready = 0;
        for (uint32_t l = 0; l < 32; ++l) if (!((done >> l) & 1u) && (dep[l] & ~done) == 0) ready |= 1u << l;
        if (!ready) { fprintf(stderr, "resolve model: no lane ready\n"); exit(1); }
        // all ready lanes copy "at once": run them in reverse lane order to expose a lane that wrongly
        // depends on a lower ready lane's output
        for (int l = 31; l >= 0; --l) if ((ready >> l) & 1u) resolve_copy_model(ob + pos[l], mlen[l], dist[l]);
        done |= ready;
        g_rounds++;
      }
    }
  }
}

int main(int argc, char** argv) {
  if (argc < 2) { fprintf(stderr, "usage: %s file.bam [max_blocks]\n", argv[0]); return 2; }
  FILE* f = fopen(argv[1], "rb");
  if (!f) { perror("open"); return 2; }
  fseek(f, 0, SEEK_END);
  size_t n = ftell(f);
  fseek(f, 0, SEEK_SET);
  std::vector<uint8_t> buf(n + 1024, 0);
  if (fread(buf.data(), 1, n, f) != n) { perror("read"); return 2; }
  fclose(f);
  size_t max_blocks = ~size_t(0);
  int fuzz = 0;
  bool all_alignments = false, expect_reject = false;
  for (int a = 2; a < argc; ++a) {
    if (!strcmp(argv[a], "--fuzz") && a + 1 < argc) fuzz = atoi(argv[++a]);
    else if (!strcmp(argv[a], "--all-alignments")) all_alignments = true;
    else if (!strcmp(argv[a], "--expect-reject")) expect_reject = true;
    else max_blocks = strtoull(argv[a], nullptr, 10);
  }
  if (fuzz || expect_reject) max_blocks = ~size_t(0);
  uint64_t rejected = 0;
  // output alignments (offset of the block's first byte mod 16): the first one uses the scalar resolve pass
  std::vector<uint32_t> aligns = {0, 9};
  if (all_alignments) { aligns.clear(); for (uint32_t a = 0; a < 16; ++a) aligns.push_back(a); }
  uint64_t fuzz_runs = 0, fuzz_failed = 0, fuzz_ok = 0, rng = 0x9E3779B97F4A7C15ull;

  InflateCounters ctr;
  static uint32_t base_lut[64];
  for (uint32_t i = 0; i < 64; ++i) base_lut[i] = base_lut_entry(i);
  std::vector<uint8_t> slab(kSlabBytes);

  std::vector<uint32_t> bitmap(kBitmapWords);
  std::vector<uint8_t> out(65536 + 64), ref(65536);
  uint64_t hist_len[260] = {0}, n_blocks = 0, total_out = 0, total_in = 0, bad = 0, resolve_tokens = 0;
  uint64_t dist_far = 0, dist_small = 0, dist_lt_len = 0, rounds_hist[34] = {0}, n_batches = 0, rounds_total = 0;
  size_t o = 0;
  while (o + 18 <= n && n_blocks < max_blocks) {
    const uint8_t* h = &buf[o];
    if (h[0] != 0x1f || h[1] != 0x8b) { fprintf(stderr, "bad magic at %zu\n", o); return 1; }
    uint32_t xlen = h[10] | (h[11] << 8);
    uint32_t bsize = h[16] | (h[17] << 8);
    size_t total = (size_t)bsize + 1;
    uint32_t isize;
    memcpy(&isize, h + total - 4, 4);
    uint32_t crc;
    memcpy(&crc, h + total - 8, 4);
    uint32_t hdr = 12 + xlen;
    uint32_t clen = (uint32_t)total - hdr - 8;
    for (int fz = 0; fz < fuzz && isize; ++fz) {
      // corrupt 1-3 bytes of a private copy of the payload (with the reader's look-ahead padding)
      std::vector<uint8_t> pay(clen + 1024, 0);
      memcpy(pay.data(), h + hdr, clen);
      int nflip = 1 + (int)(rng >> 62) % 3;
      for (int k = 0; k < nflip; ++k) {
        rng = rng * 6364136223846793005ull + 1442695040888963407ull;
        pay[(rng >> 33) % clen] ^= (uint8_t)(1u << ((rng >> 20) & 7));
      }
      BlockDesc d;
      d.in_off = (uint64_t)(uintptr_t)pay.data();
      d.out_off = 16 + (fz & 3);
      d.clen = clen;
      d.isize = isize;
      memset(out.data(), 0xAA, out.size());
      memset(bitmap.data(), 0, kBitmapWords * 4);
      Lane L;
      L.slab = slab.data();
      L.lut = base_lut;
      L.ctr = nullptr;
      L.begin_block(d, out.data(), bitmap.data());
      uint64_t steps = 0;
      while (L.state != LS_IDLE && steps < 4000000) {
        if (L.state == LS_HEADER) L.header();
        else {
          L.step();
          L.settle();
          if (L.state == LS_DECODE && L.overran()) L.end_block(kBlkBadStream);
        }
        ++steps;
      }
      if (L.state != LS_IDLE) { fprintf(stderr, "fuzz: block at %zu did not terminate\n", o); bad++; }
      uint8_t* ob = out.data() + d.out_off;
      for (int g = 1; g <= 12; ++g)
        if (ob[-g] != 0xAA || ob[isize + g - 1] != 0xAA) { fprintf(stderr, "fuzz: block at %zu wrote outside its range\n", o); bad++; break; }
      for (uint32_t w = (isize + 31) / 32 + 1; w < kBitmapWords; ++w)
        if (bitmap[w]) { fprintf(stderr, "fuzz: block at %zu marked a match beyond its size\n", o); bad++; break; }
      if (!L.err) {  // decoded "successfully": every token must be resolvable inside the block
        for (uint32_t w = 0; w < kBitmapWords; ++w)
          for (uint32_t m = bitmap[w]; m; m &= m - 1) {
            uint32_t p = w * 32 + __builtin_ctz(m);
            uint32_t tok = ob[p] | (ob[p + 1] << 8) | (ob[p + 2] << 16);
            uint32_t mlen = (tok & 255) + 3, dist = (tok >> 8) + 1;
            if (dist > p || p + mlen > isize) { fprintf(stderr, "fuzz: block at %zu holds an invalid token\n", o); bad++; w = kBitmapWords; break; }
          }
        fuzz_ok++;
      } else fuzz_failed++;
      fuzz_runs++;
    }
    if (expect_reject) {
      if (isize > 65536) { fprintf(stderr, "block at %zu: ISIZE %u > 65536\n", o, isize); return 1; }
      bool failed_everywhere = true;
      for (uint32_t a = 0; a < 16; ++a) {
        BlockDesc d;
        d.in_off = (uint64_t)(uintptr_t)(h + hdr);
        d.out_off = 16 + a;
        d.clen = clen;
        d.isize = isize;
        memset(out.data(), 0xAA, out.size());
        memset(bitmap.data(), 0, kBitmapWords * 4);
        Lane L;
        L.slab = slab.data();
        L.lut = base_lut;
        L.ctr = nullptr;
        L.begin_block(d, out.data(), bitmap.data());
        uint64_t steps = 0;
        while (L.state != LS_IDLE && steps < 4000000) {
          if (L.state == LS_HEADER) L.header();
          else {
            L.step();
            L.settle();
            if (L.state == LS_DECODE && L.overran()) L.end_block(kBlkBadStream);
          }
          ++steps;
        }
        if (L.state != LS_IDLE) { fprintf(stderr, "block at %zu: did not terminate\n", o); bad++; }
        if (!L.err) { fprintf(stderr, "block at %zu: decoded without error (output alignment %u)\n", o, a); failed_everywhere = false; }
        uint8_t* ob = out.data() + d.out_off;
        for (int g = 1; g <= 16; ++g)
          if (ob[-g] != 0xAA || ob[isize + g - 1] != 0xAA) { fprintf(stderr, "block at %zu: wrote outside its range\n", o); bad++; break; }
        for (uint32_t w = (isize + 31) / 32 + 1; w < kBitmapWords; ++w)
          if (bitmap[w]) { fprintf(stderr, "block at %zu: marked a match beyond its size\n", o); bad++; break; }
      }
      if (failed_everywhere) rejected++; else bad++;
      z_stream zs;
      memset(&zs, 0, sizeof zs);
      inflateInit2(&zs, -15);
      zs.next_in = const_cast<uint8_t*>(h + hdr);
      zs.avail_in = clen;
      zs.next_out = ref.data();
      zs.avail_out = 65536;
      const int rc = inflate(&zs, Z_FINISH);
      inflateEnd(&zs);
      if (rc == Z_STREAM_END && zs.total_out == isize) { fprintf(stderr, "block at %zu: zlib accepts it\n", o); bad++; }
      n_blocks++;
      o += total;
      continue;
    }
    if (isize && !fuzz) {
      for (uint32_t mis = 0; mis < aligns.size(); ++mis) {
        BlockDesc d;
        d.in_off = (uint64_t)(uintptr_t)(h + hdr);
        d.out_off = 16 + aligns[mis];
        d.clen = clen;
        d.isize = isize;
        memset(out.data(), 0xAA, out.size());
        memset(bitmap.data(), 0, kBitmapWords * 4);
        Lane L;
        L.slab = slab.data();
        L.lut = base_lut;
        L.ctr = mis == 0 ? &ctr : nullptr;
        L.begin_block(d, out.data(), bitmap.data());
        while (L.state != LS_IDLE) {
          if (L.state == LS_HEADER) L.header();
          else {
            L.step();
            L.settle();
            if (L.state == LS_DECODE && L.overran()) L.end_block(kBlkBadStream);
          }
        }
        if (L.err) { fprintf(stderr, "block at %zu: err %u\n", o, L.err); bad++; break; }
        // guard bytes
        uint8_t* ob = out.data() + d.out_off;
        for (int g = 1; g <= 4; ++g)
          if (ob[-g] != 0xAA || ob[isize + g - 1] != 0xAA) { fprintf(stderr, "block at %zu: wrote outside (alignment %u)\n", o, aligns[mis]); bad++; }
        // dependency depth of the resolve kernel's 32-token batches (per 1024-byte super-window)
        if (mis == 0) {
          for (uint32_t sw = 0; sw < kBitmapWords / 32; ++sw) {
            std::vector<uint32_t> ps;
            for (uint32_t w = sw * 32; w < sw * 32 + 32; ++w)
              for (uint32_t m = bitmap[w]; m; m &= m - 1) ps.push_back(w * 32 + __builtin_ctz(m));
            for (size_t base = 0; base < ps.size(); base += 32) {
              size_t nb = std::min<size_t>(32, ps.size() - base);
              uint32_t depth[32], maxd = 0;
              for (size_t j = 0; j < nb; ++j) {
                uint32_t pj = ps[base + j];
                uint32_t tok = ob[pj] | (ob[pj + 1] << 8) | (ob[pj + 2] << 16);
                uint32_t ml = (tok & 255) + 3, di = (tok >> 8) + 1;
                uint32_t slo = pj - di, shi = slo + std::min(ml, di);
                uint32_t dj = 1;
                for (size_t i = 0; i < j; ++i) {
                  uint32_t pi = ps[base + i];
                  uint32_t ti = ob[pi] | (ob[pi + 1] << 8) | (ob[pi + 2] << 16);
                  uint32_t mi = (ti & 255) + 3;
                  if (pi + mi > slo && pi < shi) dj = std::max(dj, depth[i] + 1);
                }
                depth[j] = dj;
                maxd = std::max(maxd, dj);
              }
              rounds_hist[std::min<uint32_t>(maxd, 33)]++;
              n_batches++;
              rounds_total += maxd;
            }
          }
        }
        // resolve pass: scalar in stream order for the first alignment, the warp algorithm of the kernel for the second
        if (mis != 0) resolve_block_model(ob, isize, bitmap.data());
        for (uint32_t w = 0; w < kBitmapWords && mis == 0; ++w) {
          uint32_t m = bitmap[w];
          while (m) {
            uint32_t bit = __builtin_ctz(m);
            m &= m - 1;
            uint32_t p = w * 32 + bit;
            uint32_t tok = ob[p] | (ob[p + 1] << 8) | (ob[p + 2] << 16);
            uint32_t mlen = (tok & 255) + 3, dist = (tok >> 8) + 1;
            if (mis == 0) { hist_len[mlen]++; resolve_tokens++; dist_small += dist < 4; dist_lt_len += dist < mlen; dist_far += dist >= 1024 + 258; }
            for (uint32_t k = 0; k < mlen; ++k) ob[p + k] = ob[p + k - dist];
          }
        }
        // zlib
        z_stream zs;
        memset(&zs, 0, sizeof zs);
        inflateInit2(&zs, -15);
        zs.next_in = const_cast<uint8_t*>(h + hdr);
        zs.avail_in = clen;
        zs.next_out = ref.data();
        zs.avail_out = 65536;
        int rc = inflate(&zs, Z_FINISH);
        inflateEnd(&zs);
        if (rc != Z_STREAM_END || zs.total_out != isize) { fprintf(stderr, "zlib failed at %zu\n", o); return 1; }
        if (memcmp(ref.data(), ob, isize) != 0) {
          uint32_t k = 0;
          while (ref[k] == ob[k]) ++k;
          fprintf(stderr, "block at %zu (alignment %u): MISMATCH at byte %u of %u\n", o, aligns[mis], k, isize);
          bad++;
        }
        if (crc32(0, ref.data(), isize) != crc) { fprintf(stderr, "crc mismatch at %zu\n", o); bad++; }
      }
      n_blocks++;
      total_out += isize;
      total_in += clen;
    }
    o += total;
  }
  if (expect_reject) {
    printf("reject: %llu blocks, %llu rejected, bad %llu\n", (unsigned long long)n_blocks, (unsigned long long)rejected, (unsigned long long)bad);
    return bad ? 1 : 0;
  }
  if (fuzz) {
    printf("fuzz: %llu corrupted blocks, %llu rejected, %llu decoded, bad %llu\n", (unsigned long long)fuzz_runs,
           (unsigned long long)fuzz_failed, (unsigned long long)fuzz_ok, (unsigned long long)bad);
    return bad ? 1 : 0;
  }
  printf("blocks %llu, in %llu, out %llu (ratio %.2f), bad %llu\n", (unsigned long long)n_blocks, (unsigned long long)total_in,
         (unsigned long long)total_out, (double)total_out / total_in, (unsigned long long)bad);
  printf("symbols %llu (%.3f per out byte): literals %llu (%.1f%%), matches %llu (%.1f%%), avg match len %.2f, match bytes %.1f%% of output\n",
         (unsigned long long)ctr.symbols, (double)ctr.symbols / total_out, (unsigned long long)ctr.literals, 100.0 * ctr.literals / ctr.symbols,
         (unsigned long long)ctr.matches, 100.0 * ctr.matches / ctr.symbols, (double)ctr.match_bytes / (ctr.matches ? ctr.matches : 1),
         100.0 * ctr.match_bytes / total_out);
  printf("bits per symbol %.2f\n", 8.0 * total_in / ctr.symbols);
  printf("ll code length %%:");
  for (int l = 1; l <= 15; ++l) printf(" %d:%.1f", l, 100.0 * ctr.ll_len_hist[l] / ctr.symbols);
  printf("\ndist code length %%:");
  for (int l = 1; l <= 15; ++l) printf(" %d:%.1f", l, 100.0 * ctr.d_len_hist[l] / (ctr.matches ? ctr.matches : 1));
  printf("\n");
  printf("deflate blocks per BGZF block %.2f (stored %llu, fixed %llu); symbols per deflate block %.0f\n", (double)ctr.headers / n_blocks,
         (unsigned long long)ctr.stored, (unsigned long long)ctr.fixed, (double)ctr.symbols / ctr.headers);
  printf("stores: %llu chunk + %llu edge = %.3f per output byte\n", (unsigned long long)ctr.chunk_stores, (unsigned long long)ctr.edge_stores,
         (double)(ctr.chunk_stores + ctr.edge_stores) / total_out);
  printf("dist >= 1282 (source before the resolve kernel's 1024-byte window): %.1f%% of matches\n", 100.0 * dist_far / (resolve_tokens ? resolve_tokens : 1));
  printf("dist<4: %.1f%% of matches, dist<len: %.1f%%\n", 100.0 * dist_small / (resolve_tokens ? resolve_tokens : 1), 100.0 * dist_lt_len / (resolve_tokens ? resolve_tokens : 1));
  printf("resolve batches %llu, mean dependency depth %.2f; depth histogram %%:", (unsigned long long)n_batches, (double)rounds_total / (n_batches ? n_batches : 1));
  for (int d = 1; d <= 33; ++d) if (rounds_hist[d]) printf(" %d:%.1f", d, 100.0 * rounds_hist[d] / n_batches);
  printf("\n");
  printf("warp-algorithm resolve (second alignment): %llu batches, %.2f rounds per batch\n", (unsigned long long)g_batches,
         (double)g_rounds / (g_batches ? g_batches : 1));
  printf("match length histogram (cumulative %%):");
  uint64_t cum = 0;
  for (int l = 3; l <= 258; ++l) {
    cum += hist_len[l];
    if (l <= 12 || l == 16 || l == 24 || l == 32 || l == 64 || l == 128 || l == 258) printf(" <=%d:%.1f", l, 100.0 * cum / (resolve_tokens ? resolve_tokens : 1));
  }
  printf("\n");
  return bad ? 1 : 0;
}
