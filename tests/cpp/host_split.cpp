// The C++ driver's intra-contig shard planner (ngs_b200/host/bam.hpp: read_bai, plan_shards_split, choose_shards,
// shard_bytes) on CPU.
// usage: host_split <file.bam> <first_record_voffset> <n_refs> <n_shards> [len0,len1,..]  (reference lengths; 0 without)
// prints one line per shard of plan_shards_split: first_voffset end_voffset empty lo hi contigs...
// then "split <refs...>", "anchors <voffsets...>" and "choose <contig|split> <split refs...>" (choose_shards' pick).
#include <cstdio>
#include <cstdlib>

#include "../../ngs_b200/host/bam.hpp"

using namespace ngs;

int main(int argc, char** argv) {
  if (argc < 5) return 2;
  try {
    MappedFile file(argv[1]);
    BaiIndex bai = read_bai(std::string(argv[1]) + ".bai");
    BamHeader h;
    h.first_record_voffset = strtoull(argv[2], nullptr, 10);
    h.reference_sequences.resize(strtoul(argv[3], nullptr, 10));
    if (argc > 5) {
      char* p = argv[5];
      for (auto& rs : h.reference_sequences) { rs.length = (uint32_t)strtoul(p, &p, 10); if (*p == ',') ++p; }
    }
    const uint32_t n = (uint32_t)atoi(argv[4]);
    const ShardPlan plan = plan_shards_split(h, bai, n, file.size());
    for (const Shard& s : plan.shards) {
      uint64_t lo = 0, hi = 0;
      if (!s.empty) shard_bytes(s, file.data(), file.size(), &lo, &hi);
      printf("%llu %llu %d %llu %llu", (unsigned long long)s.first_voffset, (unsigned long long)s.end_voffset, s.empty ? 1 : 0, (unsigned long long)lo, (unsigned long long)hi);
      for (uint32_t c : s.contigs) printf(" %u", c);
      printf("\n");
    }
    printf("split");
    for (uint32_t c : plan.split) printf(" %u", c);
    printf("\nanchors");
    for (uint64_t v : bai_anchors(bai)) printf(" %llu", (unsigned long long)v);
    const ShardPlan pick = choose_shards(h, bai, n, file.size());
    printf("\nchoose %s", pick.split_plan ? "split" : "contig");
    for (uint32_t c : pick.split) printf(" %u", c);
    printf("\n");
  } catch (const std::exception& e) {
    printf("error: %s\n", e.what());
  }
  return 0;
}
