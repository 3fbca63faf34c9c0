// The C++ driver's CSI reader (ngs_b200/host/bam.hpp: parse_csi) and the shard planners it feeds (plan_shards,
// plan_shards_split, bai_anchors) on CPU.
// usage: host_csi <file.bam> <index> <csi|bai> <first_record_voffset> <n_refs> <n_shards>
//   csi: <index> is an UNCOMPRESSED .csi payload, read by parse_csi with <n_refs> as the BAM header's reference count;
//   bai: <index> is a .bai, read by read_bai (the same planner input, for comparison).
// prints "ref has_extent ref_beg ref_end n_mapped n_unmapped" per reference, "anchors <voffsets...>", one
// "contig first_voffset end_voffset empty contigs..." line per shard of plan_shards, one
// "shard first_voffset end_voffset empty lo hi contigs..." line per shard of plan_shards_split, then "split <refs...>";
// or "error: <message>".
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../ngs_b200/host/bam.hpp"

using namespace ngs;

int main(int argc, char** argv) {
  if (argc < 7) return 2;
  try {
    MappedFile file(argv[1]);
    const size_t n_refs = strtoul(argv[5], nullptr, 10);
    BaiIndex idx;
    if (!strcmp(argv[3], "csi")) {
      MappedFile payload(argv[2]);
      idx = parse_csi(payload.data(), payload.size(), argv[2], n_refs);
    } else {
      idx = read_bai(argv[2]);
    }
    BamHeader h;
    h.first_record_voffset = strtoull(argv[4], nullptr, 10);
    h.reference_sequences.resize(n_refs);
    const uint32_t n = (uint32_t)atoi(argv[6]);
    for (const BaiReference& r : idx.refs)
      printf("ref %d %llu %llu %llu %llu\n", r.has_extent ? 1 : 0, (unsigned long long)r.ref_beg, (unsigned long long)r.ref_end,
             (unsigned long long)r.n_mapped, (unsigned long long)r.n_unmapped);
    printf("anchors");
    for (uint64_t v : bai_anchors(idx)) printf(" %llu", (unsigned long long)v);
    printf("\n");
    for (const Shard& s : plan_shards(h, idx, n, file.size())) {
      printf("contig %llu %llu %d", (unsigned long long)s.first_voffset, (unsigned long long)s.end_voffset, s.empty ? 1 : 0);
      for (uint32_t c : s.contigs) printf(" %u", c);
      printf("\n");
    }
    const ShardPlan plan = plan_shards_split(h, idx, n, file.size());
    for (const Shard& s : plan.shards) {
      uint64_t lo = 0, hi = 0;
      if (!s.empty) shard_bytes(s, file.data(), file.size(), &lo, &hi);
      printf("shard %llu %llu %d %llu %llu", (unsigned long long)s.first_voffset, (unsigned long long)s.end_voffset, s.empty ? 1 : 0,
             (unsigned long long)lo, (unsigned long long)hi);
      for (uint32_t c : s.contigs) printf(" %u", c);
      printf("\n");
    }
    printf("split");
    for (uint32_t c : plan.split) printf(" %u", c);
    printf("\n");
  } catch (const std::exception& e) {
    printf("error: %s\n", e.what());
  }
  return 0;
}
