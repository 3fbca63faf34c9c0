// bamshuffle — writes the records of a BAM again in a seeded random order (the header as it is), for measuring
// `qc --cuda-any-order` on a file of realistic size (tools/any_order_bench.py).  Seed 0 keeps the file's order; with parts > 1
// the records go to that many files <out>.<k>.bam of consecutive records, each with the header, for measuring `qc --cuda-also`
// (tools/multi_file_bench.py).  Blocks are inflated and deflated on all threads; the records are packed into BGZF blocks of
// 0xFF00 bytes, so they straddle block boundaries.
//   bamshuffle <in.bam> <out.bam> [seed] [zlib level] [threads] [parts]
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <random>
#include <string>
#include <thread>
#include <vector>

namespace {

std::vector<uint8_t> slurp(const char* path) {
  FILE* f = fopen(path, "rb");
  if (!f) { fprintf(stderr, "cannot open %s\n", path); exit(1); }
  fseek(f, 0, SEEK_END);
  std::vector<uint8_t> b((size_t)ftell(f));
  fseek(f, 0, SEEK_SET);
  if (fread(b.data(), 1, b.size(), f) != b.size()) { fprintf(stderr, "short read on %s\n", path); exit(1); }
  fclose(f);
  return b;
}

uint32_t rd32(const uint8_t* p) { uint32_t v; memcpy(&v, p, 4); return v; }

template <class F>
void parallel_for(size_t n, int threads, F f) {
  std::atomic<size_t> next{0};
  std::vector<std::thread> ts;
  for (int t = 0; t < threads; ++t)
    ts.emplace_back([&] { for (size_t i; (i = next.fetch_add(1)) < n;) f(i); });
  for (auto& t : ts) t.join();
}

// one BGZF block of payload [p, p + n) at `level` (n <= 0xFF00)
std::vector<uint8_t> deflate_block(const uint8_t* p, size_t n, int level) {
  std::vector<uint8_t> out(18 + compressBound((uLong)n) + 8);
  z_stream zs{};
  if (deflateInit2(&zs, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) { fprintf(stderr, "deflateInit2\n"); exit(1); }
  zs.next_in = const_cast<uint8_t*>(p);
  zs.avail_in = (uInt)n;
  zs.next_out = out.data() + 18;
  zs.avail_out = (uInt)(out.size() - 26);
  if (deflate(&zs, Z_FINISH) != Z_STREAM_END) { fprintf(stderr, "deflate\n"); exit(1); }
  const size_t clen = zs.total_out;
  deflateEnd(&zs);
  static const uint8_t hdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
  memcpy(out.data(), hdr, 16);
  const uint16_t bsize = (uint16_t)(26 + clen - 1);
  const uint32_t crc = (uint32_t)crc32(crc32(0, nullptr, 0), p, (uInt)n), isize = (uint32_t)n;
  memcpy(out.data() + 16, &bsize, 2);
  memcpy(out.data() + 18 + clen, &crc, 4);
  memcpy(out.data() + 22 + clen, &isize, 4);
  out.resize(26 + clen);
  return out;
}

}  // namespace

int main(int argc, char** argv) {
  if (argc < 3) { fprintf(stderr, "usage: bamshuffle <in.bam> <out.bam> [seed] [zlib level] [threads] [parts]\n"); return 2; }
  const uint64_t seed = argc > 3 ? strtoull(argv[3], nullptr, 0) : 1;
  const int level = argc > 4 ? atoi(argv[4]) : 1;
  const int threads = argc > 5 ? atoi(argv[5]) : (int)std::max(1u, std::thread::hardware_concurrency());
  const size_t parts = argc > 6 ? std::max(1, atoi(argv[6])) : 1;
  const std::vector<uint8_t> in = slurp(argv[1]);
  // blocks, then their inflated bytes side by side
  std::vector<size_t> coff, uoff{0};
  for (size_t o = 0; o + 18 <= in.size();) {
    const size_t bsize = (size_t)(in[o + 16] | (in[o + 17] << 8)) + 1;
    if (o + bsize > in.size()) { fprintf(stderr, "truncated block at %zu\n", o); return 1; }
    coff.push_back(o);
    uoff.push_back(uoff.back() + rd32(&in[o + bsize - 4]));
    o += bsize;
  }
  std::vector<uint8_t> data(uoff.back());
  parallel_for(coff.size(), threads, [&](size_t k) {
    const size_t o = coff[k], bsize = (size_t)(in[o + 16] | (in[o + 17] << 8)) + 1, xlen = in[o + 10] | (in[o + 11] << 8);
    z_stream zs{};
    inflateInit2(&zs, -15);
    zs.next_in = const_cast<uint8_t*>(&in[o + 12 + xlen]);
    zs.avail_in = (uInt)(bsize - 12 - xlen - 8);
    zs.next_out = data.data() + uoff[k];
    zs.avail_out = (uInt)(uoff[k + 1] - uoff[k]);
    const int rc = inflate(&zs, Z_FINISH);
    inflateEnd(&zs);
    if (rc != Z_STREAM_END) { fprintf(stderr, "inflate failed in block at %zu\n", o); exit(1); }
  });
  // header: magic, l_text, text, n_ref, references
  size_t h = 8 + rd32(&data[4]);
  const uint32_t n_ref = rd32(&data[h]);
  h += 4;
  for (uint32_t c = 0; c < n_ref; ++c) h += 4 + rd32(&data[h]) + 4;
  std::vector<size_t> rec;
  for (size_t o = h; o + 4 <= data.size(); o += 4 + rd32(&data[o])) rec.push_back(o);
  if (seed) {
    std::mt19937_64 rng(seed);
    for (size_t i = rec.size(); i > 1; --i) std::swap(rec[i - 1], rec[std::uniform_int_distribution<size_t>(0, i - 1)(rng)]);
  }
  // the header in blocks of its own, as bamgen and samtools write it
  std::vector<std::vector<uint8_t>> hdr_blocks;
  for (size_t o = 0; o < h; o += 0xFF00) hdr_blocks.push_back(deflate_block(data.data() + o, std::min<size_t>(0xFF00, h - o), level));
  static const uint8_t kEof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  size_t n_blocks = 0;
  for (size_t k = 0; k < parts; ++k) {
    const size_t r0 = rec.size() * k / parts, r1 = rec.size() * (k + 1) / parts;
    size_t bytes = 0;
    for (size_t i = r0; i < r1; ++i) bytes += 4 + rd32(&data[rec[i]]);
    std::vector<uint8_t> stream(bytes);
    size_t w = 0;
    for (size_t i = r0; i < r1; ++i) {
      const size_t n = 4 + rd32(&data[rec[i]]);
      memcpy(stream.data() + w, &data[rec[i]], n);
      w += n;
    }
    const size_t n_out = (stream.size() + 0xFF00 - 1) / 0xFF00;
    std::vector<std::vector<uint8_t>> blocks(n_out);
    parallel_for(n_out, threads, [&](size_t j) {
      blocks[j] = deflate_block(stream.data() + j * 0xFF00, std::min<size_t>(0xFF00, stream.size() - j * 0xFF00), level);
    });
    const std::string path = parts == 1 ? std::string(argv[2]) : std::string(argv[2]) + "." + std::to_string(k) + ".bam";
    FILE* f = fopen(path.c_str(), "wb");
    if (!f) { fprintf(stderr, "cannot create %s\n", path.c_str()); return 1; }
    bool ok = true;
    for (const auto& b : hdr_blocks) ok = ok && fwrite(b.data(), 1, b.size(), f) == b.size();
    for (const auto& b : blocks) ok = ok && fwrite(b.data(), 1, b.size(), f) == b.size();
    ok = ok && fwrite(kEof, 1, 28, f) == 28;
    if (fclose(f) || !ok) { fprintf(stderr, "write error on %s\n", path.c_str()); return 1; }
    n_blocks += n_out;
  }
  fprintf(stderr, "%zu records, %zu blocks, %zu file(s)\n", rec.size(), n_blocks, parts);
  return 0;
}
