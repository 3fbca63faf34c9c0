// The C++ driver's cuts without an index (ngs_b200/host/bam.hpp: next_block_start, plan_shards_unindexed) on CPU, with a
// record finder backed by the truth (every record start, found by the test with zlib) instead of the GPU one.
// usage: host_unindexed blocks <file.bam>
//          prints every block start next_block_start finds, one per line
//        host_unindexed plan <file.bam> <first_record_voffset> <n_shards> <truth file: "voffset ref_id" per record>
//          prints one line per shard (first_voffset end_voffset empty), then "split <refs...>", "dropped <n>" and
//          "windows <largest window the finder was offered, in bytes>"
#include <cstdio>
#include <cstdlib>

#include "../../ngs_b200/host/bam.hpp"

using namespace ngs;

int main(int argc, char** argv) {
  if (argc < 3) return 2;
  try {
    MappedFile file(argv[2]);
    const std::string mode = argv[1];
    if (mode == "blocks") {
      for (uint64_t q = next_block_start(file.data(), file.size(), 0); q < file.size(); q = next_block_start(file.data(), file.size(), q + 1))
        printf("%llu\n", (unsigned long long)q);
      return 0;
    }
    if (mode != "plan" || argc < 6) return 2;
    BamHeader h;
    h.first_record_voffset = strtoull(argv[3], nullptr, 10);
    std::vector<std::pair<uint64_t, int32_t>> truth;
    FILE* f = fopen(argv[5], "r");
    if (!f) return 2;
    unsigned long long v;
    int r;
    while (fscanf(f, "%llu %d", &v, &r) == 2) truth.push_back({v, r});
    fclose(f);
    size_t widest = 0;
    // the first record that starts in one of the window's blocks
    FindRecord find = [&](const uint8_t*, size_t n, uint64_t off, uint64_t* voff, int32_t* ref) {
      widest = std::max(widest, n);
      *voff = 0;
      *ref = -1;
      auto it = std::lower_bound(truth.begin(), truth.end(), std::make_pair(off << 16, INT32_MIN));
      if (it != truth.end() && (it->first >> 16) < off + n) { *voff = it->first; *ref = it->second; }
    };
    const ShardPlan plan = plan_shards_unindexed(h, file.data(), file.size(), (uint32_t)atoi(argv[4]), find);
    for (const Shard& s : plan.shards)
      printf("%llu %llu %d\n", (unsigned long long)s.first_voffset, (unsigned long long)s.end_voffset, s.empty ? 1 : 0);
    printf("split");
    for (uint32_t c : plan.split) printf(" %u", c);
    printf("\ndropped %u\nwindows %zu\n", plan.dropped, widest);
  } catch (const std::exception& e) {
    printf("error: %s\n", e.what());
  }
  return 0;
}
