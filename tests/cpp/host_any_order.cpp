// The C++ driver's plan for records in any order (ngs_b200/host/bam.hpp: plan_shards_any_order) on CPU, with a record finder
// backed by the truth (every record start, found by the test with zlib) instead of the GPU one.
// usage: host_any_order <file.bam> <first_record_voffset> <n_ref> <n_shards> <truth file: "voffset ref_id" per record>
//          prints one line per shard (first_voffset end_voffset empty), then "split <refs...>" and "dropped <n>"
#include <cstdio>
#include <cstdlib>

#include "../../ngs_b200/host/bam.hpp"

using namespace ngs;

int main(int argc, char** argv) {
  if (argc < 6) return 2;
  try {
    MappedFile file(argv[1]);
    BamHeader h;
    h.first_record_voffset = strtoull(argv[2], nullptr, 10);
    h.reference_sequences.resize((size_t)atoi(argv[3]));
    std::vector<std::pair<uint64_t, int32_t>> truth;
    FILE* f = fopen(argv[5], "r");
    if (!f) return 2;
    unsigned long long v;
    int r;
    while (fscanf(f, "%llu %d", &v, &r) == 2) truth.push_back({v, r});
    fclose(f);
    // the first record that starts in one of the window's blocks
    FindRecord find = [&](const uint8_t*, size_t n, uint64_t off, uint64_t* voff, int32_t* ref) {
      *voff = 0;
      *ref = -1;
      auto it = std::lower_bound(truth.begin(), truth.end(), std::make_pair(off << 16, INT32_MIN));
      if (it != truth.end() && (it->first >> 16) < off + n) { *voff = it->first; *ref = it->second; }
    };
    const ShardPlan plan = plan_shards_any_order(h, file.data(), file.size(), (uint32_t)atoi(argv[4]), find);
    for (const Shard& s : plan.shards)
      printf("%llu %llu %d\n", (unsigned long long)s.first_voffset, (unsigned long long)s.end_voffset, s.empty ? 1 : 0);
    printf("split");
    for (uint32_t c : plan.split) printf(" %u", c);
    printf("\ndropped %u\n", plan.dropped);
  } catch (const std::exception& e) {
    printf("error: %s\n", e.what());
  }
  return 0;
}
