// The C++ driver's plan for several files of one sample (ngs_b200/host/bam.hpp: check_same_dictionary, assign_files,
// devices_per_file, plan_files) on CPU, with a record finder backed by the truth instead of the GPU one.
// usage: host_multi_file dict <a.txt> <b.txt>          (one "name length" per line; prints "ok" or "error: <message>")
//        host_multi_file assign <n_dev> <bytes...>     (one line per device: its files in the order it runs them)
//        host_multi_file split <n_dev> <bytes...>      (the devices of every file)
//        host_multi_file plan <n_dev> <n_ref> {<file.bam> <first_record_voffset> <truth: "voffset ref_id" per record>}...
//          (one line per device: "file first_voffset end_voffset empty" per queued part; then "cut <0|1>" and "dropped <n>")
#include <cstdio>
#include <cstdlib>
#include <memory>

#include "../../ngs_b200/host/bam.hpp"

using namespace ngs;

static std::vector<ReferenceSequence> read_dict(const char* path) {
  std::vector<ReferenceSequence> v;
  std::ifstream f(path);
  std::string name;
  uint32_t len;
  while (f >> name >> len) v.push_back({name, len});
  return v;
}

int main(int argc, char** argv) {
  if (argc < 3) return 2;
  const std::string mode = argv[1];
  try {
    if (mode == "dict") {
      check_same_dictionary(argv[2], read_dict(argv[2]), argv[3], read_dict(argv[3]));
      printf("ok\n");
      return 0;
    }
    const uint32_t n_dev = (uint32_t)atoi(argv[2]);
    if (mode == "assign" || mode == "split") {
      std::vector<uint64_t> bytes;
      for (int i = 3; i < argc; ++i) bytes.push_back(strtoull(argv[i], nullptr, 10));
      if (mode == "split") {
        for (uint32_t n : devices_per_file(bytes, n_dev)) printf("%u ", n);
        printf("\n");
        return 0;
      }
      for (const auto& q : assign_files(bytes, n_dev)) {
        for (uint32_t f : q) printf("%u ", f);
        printf("\n");
      }
      return 0;
    }
    if (mode != "plan") return 2;
    const size_t n_ref = (size_t)atoi(argv[3]);
    std::vector<std::unique_ptr<MappedFile>> files;
    std::vector<BamHeader> headers;
    std::vector<const uint8_t*> data;
    std::vector<uint64_t> sizes;
    std::vector<std::vector<std::pair<uint64_t, int32_t>>> truth;
    for (int i = 4; i + 2 < argc; i += 3) {
      files.push_back(std::make_unique<MappedFile>(argv[i]));
      BamHeader h;
      h.first_record_voffset = strtoull(argv[i + 1], nullptr, 10);
      h.reference_sequences.resize(n_ref);
      headers.push_back(h);
      data.push_back(files.back()->data());
      sizes.push_back(files.back()->size());
      truth.emplace_back();
      FILE* f = fopen(argv[i + 2], "r");
      if (!f) return 2;
      unsigned long long v;
      int r;
      while (fscanf(f, "%llu %d", &v, &r) == 2) truth.back().push_back({v, r});
      fclose(f);
    }
    // the first record that starts in one of the window's blocks, of the file the window was cut from
    FindRecord find = [&](const uint8_t* p, size_t n, uint64_t off, uint64_t* voff, int32_t* ref) {
      *voff = 0;
      *ref = -1;
      size_t k = 0;
      while (k < data.size() && !(p >= data[k] && p < data[k] + sizes[k])) ++k;
      if (k == data.size()) return;
      auto it = std::lower_bound(truth[k].begin(), truth[k].end(), std::make_pair(off << 16, INT32_MIN));
      if (it != truth[k].end() && (it->first >> 16) < off + n) { *voff = it->first; *ref = it->second; }
    };
    const FilePlan plan = plan_files(headers, data, sizes, n_dev, find);
    for (const auto& q : plan.queues) {
      for (const FilePart& p : q)
        printf("%u %llu %llu %d ", p.file, (unsigned long long)p.shard.first_voffset, (unsigned long long)p.shard.end_voffset, p.shard.empty ? 1 : 0);
      printf("\n");
    }
    printf("cut %d\ndropped %u\n", plan.cut ? 1 : 0, plan.dropped);
  } catch (const std::exception& e) {
    printf("error: %s\n", e.what());
  }
  return 0;
}
