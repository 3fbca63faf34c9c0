// Drives ngs_b200/host/read_groups.hpp on CPU.  usage:
//   host_read_groups ids <header text file> <path>      the @RG IDs, one per line, or "error: <message>"
//   host_read_groups union <file> [<file> ..]           the union of the IDs of several header texts
//   host_read_groups escape <hex> [<hex> ..]            the file-name form of each ID (given as hex bytes)
//   host_read_groups only <facet>                       "ok" or "error: <message>" for --only <facet>
//   host_read_groups group <g> <dir> <prefix>           group g's results JSON from the test double's integers
//                                                       (fake_engine.cpp; ngsq_select_read_group below)
#include <fstream>
#include <iostream>
#include <sstream>

#include "../../ngs_b200/host/read_groups.hpp"

using namespace ngs;

extern "C" int ngsq_select_read_group(ngsq_engine*, int32_t) { return 0; }  // the double serves one group's integers

static std::string slurp(const char* p) {
  std::ifstream f(p, std::ios::binary);
  std::stringstream ss;
  ss << f.rdbuf();
  return ss.str();
}

int main(int argc, char** argv) {
  if (argc < 2) return 2;
  const std::string mode = argv[1];
  try {
    if (mode == "ids") {
      for (const auto& id : read_group_ids(slurp(argv[2]), argv[3])) std::cout << id << "\n";
    } else if (mode == "union") {
      std::vector<std::vector<std::string>> per;
      for (int i = 2; i < argc; ++i) per.push_back(read_group_ids(slurp(argv[i]), argv[i]));
      for (const auto& id : union_read_group_ids(per)) std::cout << id << "\n";
    } else if (mode == "escape") {
      for (int i = 2; i < argc; ++i) {
        std::string id;
        for (const char* h = argv[i]; h[0] && h[1]; h += 2) id += (char)std::stoi(std::string(h, 2), nullptr, 16);
        std::cout << escape_read_group_id(id) << "\n";
      }
    } else if (mode == "only") {
      check_read_group_facet(std::string(argv[2]));
      std::cout << "ok\n";
    } else if (mode == "group") {
      auto genome = get_reference_genome("GRCh38_no_alt_AnalysisSet");
      ngsq_engine* root = reinterpret_cast<ngsq_engine*>(1);
      read_group_results(root, std::stoi(argv[2]), *genome, std::nullopt).write(argv[4], argv[3]);
    } else {
      return 2;
    }
  } catch (const std::exception& ex) {
    std::cout << "error: " << ex.what() << "\n";
  }
  return 0;
}
