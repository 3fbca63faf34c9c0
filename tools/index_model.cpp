// CPU model of the BAI / CSI index kernel (test tooling; NOT part of the product library): runs the per-record functions the
// CUDA kernel calls (ngs_b200/csrc/index.cuh: index_record, index_windows) over every
// record of a BAM, with the virtual offsets the engine gives them.
//   g++ -O2 -std=c++17 -o /tmp/index_model tools/index_model.cpp -lz
//   /tmp/index_model file.bam   -> per record "ref pos bin beg end placed unmapped voff w_lo w_hi", or a last line "error <kind>"
//   /tmp/index_model file.bam --csi MIN_SHIFT DEPTH   -> the same with the CSI key and windows of 2^MIN_SHIFT bases
#include <zlib.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../ngs_b200/csrc/index.cuh"

using namespace ngsq;

static std::vector<uint8_t> slurp(const char* path) {
  FILE* f = fopen(path, "rb");
  if (!f) { perror(path); exit(2); }
  fseek(f, 0, SEEK_END);
  long n = ftell(f);
  fseek(f, 0, SEEK_SET);
  std::vector<uint8_t> b(n);
  if (n && fread(b.data(), 1, n, f) != (size_t)n) { perror("read"); exit(2); }
  fclose(f);
  return b;
}

int main(int argc, char** argv) {
  const bool csi = argc == 5 && !strcmp(argv[2], "--csi");
  if (argc != 2 && !csi) { fprintf(stderr, "usage: %s file.bam [--csi MIN_SHIFT DEPTH]\n", argv[0]); return 2; }
  const uint32_t min_shift = csi ? (uint32_t)atoi(argv[3]) : kIxWindowShift, depth = csi ? (uint32_t)atoi(argv[4]) : 5;
  std::vector<uint8_t> bam = slurp(argv[1]);
  // inflated stream + file offset of the block that holds each of its bytes (non-empty blocks only, like the engine)
  std::vector<uint8_t> s;
  std::vector<uint64_t> blk_start, blk_coff;
  for (size_t o = 0; o + 18 <= bam.size();) {
    const size_t total = (size_t)(bam[o + 16] | (bam[o + 17] << 8)) + 1;
    uint32_t isize;
    memcpy(&isize, &bam[o + total - 4], 4);
    const size_t at = s.size();
    if (isize) { blk_start.push_back(at); blk_coff.push_back(o); }
    s.resize(at + isize);
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    inflateInit2(&zs, -15);
    zs.next_in = &bam[o + 18];
    zs.avail_in = (uInt)(total - 26);
    zs.next_out = s.data() + at;
    zs.avail_out = isize;
    if (isize && inflate(&zs, Z_FINISH) != Z_STREAM_END) { fprintf(stderr, "inflate failed\n"); return 2; }
    inflateEnd(&zs);
    o += total;
  }
  auto voff = [&](uint64_t x) {
    size_t lo = 0, hi = blk_start.size();
    while (hi - lo > 1) { const size_t mid = (lo + hi) / 2; if (blk_start[mid] <= x) lo = mid; else hi = mid; }
    return (blk_coff[lo] << 16) | (x - blk_start[lo]);
  };
  uint32_t l_text, n_ref;
  memcpy(&l_text, &s[4], 4);
  size_t p = 8 + l_text;
  memcpy(&n_ref, &s[p], 4);
  p += 4;
  for (uint32_t c = 0; c < n_ref; ++c) {
    uint32_t ln;
    memcpy(&ln, &s[p], 4);
    p += 8 + ln;
  }
  while (p + 36 <= s.size()) {
    uint32_t bs;
    memcpy(&bs, &s[p], 4);
    IndexKey k;
    const uint32_t err = index_record(&s[p], (int32_t)n_ref, &k, csi, min_shift, depth);
    if (err) { printf("error %u\n", err); return 0; }
    uint32_t w_lo = 0, w_hi = 0;
    if (k.placed) index_windows(k, &w_lo, &w_hi, min_shift);
    printf("%d %d %u %llu %llu %u %u %llu %u %u\n", k.ref, k.pos, k.bin, (unsigned long long)k.beg, (unsigned long long)k.end, k.placed,
           k.unmapped, (unsigned long long)voff(p), w_lo, w_hi);
    p += 4 + (size_t)bs;
  }
  return 0;
}
