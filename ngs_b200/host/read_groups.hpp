// `qc --cuda-by-read-group`: the @RG IDs of the header(s), the per-group file names, and one results JSON per read group from
// the engine's group tables (NGSQ_F_READ_GROUPS, ngsq_select_read_group).  The four record facets of a group are the host
// facets of facets.hpp fed with that group's integers; Coverage, Edits and Genomic Features stay the sample's.
#pragma once
#include <zlib.h>

#include <cstring>
#include <optional>
#include <set>
#include <stdexcept>
#include <string>
#include <vector>

#include "facets.hpp"

namespace ngs {

constexpr uint32_t kMaxReadGroups = 65534;  // ngsq_set_read_groups

// The SAM header text of a BAM, inflated on the host block by block until its l_text bytes are in: `--cuda-by-read-group`
// checks the @RG lines before any device work.
inline std::string bam_header_text(const uint8_t* bam, size_t size, const std::string& path) {
  std::string out;
  std::vector<uint8_t> buf(65536);
  for (size_t off = 0; off + 18 <= size;) {
    const uint8_t* p = bam + off;
    if (p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) break;
    const uint32_t xlen = p[10] | (p[11] << 8);
    uint32_t bsize = 0;
    for (uint32_t q = 0; q + 4 <= xlen && 12 + q + 6 <= size - off;) {
      const uint8_t* f = p + 12 + q;
      const uint32_t slen = f[2] | (f[3] << 8);
      if (f[0] == 'B' && f[1] == 'C' && slen == 2) bsize = f[4] | (f[5] << 8);
      q += 4 + slen;
    }
    const size_t total = (size_t)bsize + 1;
    if (!bsize || total < 12 + xlen + 8 || off + total > size) break;
    z_stream zs{};
    if (inflateInit2(&zs, -15) != Z_OK) break;
    zs.next_in = const_cast<uint8_t*>(p + 12 + xlen);
    zs.avail_in = (uInt)(total - 12 - xlen - 8);
    zs.next_out = buf.data();
    zs.avail_out = (uInt)buf.size();
    const int rc = inflate(&zs, Z_FINISH);
    const size_t got = zs.total_out;
    inflateEnd(&zs);
    if (rc != Z_STREAM_END) break;
    out.append((const char*)buf.data(), got);
    off += total;
    if (out.size() >= 8) {
      if (out.compare(0, 4, std::string("BAM\1", 4)) != 0) throw std::runtime_error("could not open " + path + ": not a BAM file (bad magic)");
      uint32_t l_text;
      memcpy(&l_text, out.data() + 4, 4);
      if (out.size() >= 8 + (size_t)l_text) return out.substr(8, l_text);
    }
  }
  throw std::runtime_error("could not open " + path + ": malformed or truncated BAM header");
}

// The ID: of every @RG line of a SAM header text, in header order.  Refuses a header without @RG lines, an @RG line without
// an ID: field (or with an empty one) and an ID declared twice: the groups would not be defined.
inline std::vector<std::string> read_group_ids(const std::string& text, const std::string& path) {
  std::vector<std::string> ids;
  std::set<std::string> seen;
  size_t pos = 0;
  while (pos < text.size()) {
    size_t eol = text.find('\n', pos);
    if (eol == std::string::npos) eol = text.size();
    std::string line = text.substr(pos, eol - pos);
    pos = eol + 1;
    if (!line.empty() && line.back() == '\r') line.pop_back();
    if (line.compare(0, 4, "@RG\t") != 0 && line != "@RG") continue;
    std::optional<std::string> id;
    for (size_t f = 3; f < line.size();) {
      size_t end = line.find('\t', f + 1);
      if (end == std::string::npos) end = line.size();
      const std::string field = line.substr(f + 1, end - f - 1);
      if (field.compare(0, 3, "ID:") == 0) { id = field.substr(3); break; }
      f = end;
    }
    if (!id || id->empty()) throw std::runtime_error("--cuda-by-read-group: an @RG line of " + path + " has no ID: \"" + line + "\"");
    if (!seen.insert(*id).second) throw std::runtime_error("--cuda-by-read-group: the read group ID \"" + *id + "\" is declared twice in the header of " + path);
    ids.push_back(*id);
  }
  if (ids.empty()) throw std::runtime_error("--cuda-by-read-group: the header of " + path + " has no @RG line");
  return ids;
}

// Several files of one sample (`--cuda-also`): the union of their IDs, first file first, each ID once (a run cut into chunk
// files repeats its read groups).
inline std::vector<std::string> union_read_group_ids(const std::vector<std::vector<std::string>>& per_file) {
  std::vector<std::string> out;
  std::set<std::string> seen;
  for (const auto& ids : per_file)
    for (const auto& id : ids)
      if (seen.insert(id).second) out.push_back(id);
  if (out.size() > kMaxReadGroups)
    throw std::runtime_error("--cuda-by-read-group: " + std::to_string(out.size()) + " read groups, at most " + std::to_string(kMaxReadGroups));
  return out;
}

// The ID in a file name: every byte outside [A-Za-z0-9._-], and '%' itself, as %XX (upper-case hex).  Distinct IDs give
// distinct names, and no ID can leave the output directory.
inline std::string escape_read_group_id(const std::string& id) {
  static const char hex[] = "0123456789ABCDEF";
  std::string out;
  for (unsigned char c : id) {
    const bool keep = (c >= 'A' && c <= 'Z') || (c >= 'a' && c <= 'z') || (c >= '0' && c <= '9') || c == '.' || c == '_' || c == '-';
    if (keep) out += (char)c;
    else { out += '%'; out += hex[c >> 4]; out += hex[c & 15]; }
  }
  return out;
}

// The output prefixes of group g (0..n-1) and of the ungrouped records
inline std::string read_group_prefix(const std::string& prefix, const std::string& id) { return prefix + ".read_group." + escape_read_group_id(id); }
inline std::string no_read_group_prefix(const std::string& prefix) { return prefix + ".no_read_group"; }

// --only with a facet that has no per-group results is refused (nothing would be written per group)
inline void check_read_group_facet(const std::optional<std::string>& only) {
  if (!only) return;
  for (const char* f : {"Coverage", "Edits", "Genomic Features"})
    if (eq_ignore_ascii_case(f, *only))
      throw std::runtime_error(std::string("--cuda-by-read-group cannot be combined with --only ") + *only +
                               ": the per-group results hold General, Template Length, GC Content and Quality Score only");
}

// The results of group g of a finished engine: the record facets `--only` selects, fed with the group's integers.
inline Results read_group_results(ngsq_engine* e, int32_t g, const ReferenceGenome& genome, const std::optional<std::string>& only) {
  check(e, ngsq_select_read_group(e, g));
  FacetSet facets = get_qc_facets(genome, only);
  Results results;
  for (auto& f : facets.record_based) { f->ingest(e); f->summarize(); f->aggregate(results); }
  check(e, ngsq_select_read_group(e, -1));
  return results;
}

// Writes <dir>/<prefix>.read_group.<ID>.results.json for every ID, and <dir>/<prefix>.no_read_group.results.json when some
// records belong to no declared group; returns the number of those records.
inline uint64_t write_read_group_results(ngsq_engine* e, const std::vector<std::string>& ids, const ReferenceGenome& genome,
                                         const std::optional<std::string>& only, const std::string& prefix, const std::string& dir) {
  for (size_t g = 0; g < ids.size(); ++g) read_group_results(e, (int32_t)g, genome, only).write(read_group_prefix(prefix, ids[g]), dir);
  uint64_t general[34];
  check(e, ngsq_select_read_group(e, (int32_t)ids.size()));
  check(e, ngsq_get_general(e, general));
  check(e, ngsq_select_read_group(e, -1));
  if (general[0]) read_group_results(e, (int32_t)ids.size(), genome, only).write(no_read_group_prefix(prefix), dir);
  return general[0];
}

}  // namespace ngs
