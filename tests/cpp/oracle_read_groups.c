/* TEST INFRASTRUCTURE: the oracle's pass 1 (oracle/ngsqc_oracle.c, compiled into this file unchanged) restricted to one read
 * group, for `qc --cuda-by-read-group` (NGSQ_F_READ_GROUPS).  The record-based facets take only the records that pass the
 * filter; `-n` counts every record, as in the engine.  Which group a record belongs to restates htslib's bam_aux_get: the
 * FIRST aux field tagged RG decides; a type other than Z, or a value no declared ID matches byte for byte, makes the record
 * ungrouped.  A malformed aux field in front of it (unknown type, no NUL, a field that runs past the record) fails the run.
 * The results are read with the oracle's own getters (oracle_get_general, ...). */
#include "../../oracle/ngsqc_oracle.c"

/* bytes of the inflated stream consumed so far (empty blocks count nothing) */
static uint64_t rg_stream_pos(const bgzf_t* r) { return r->inflated_total - (r->cur_len - r->cur_off); }

/* 0..n_ids-1: the group; n_ids: ungrouped; -1: malformed aux field (g_err set) */
static int64_t rg_group(const uint8_t* a, const uint8_t* end, const char* const* ids, uint32_t n_ids) {
  while (a < end) {
    if (end - a < 3) { snprintf(g_err, sizeof g_err, "aux field header runs past the record"); return -1; }
    uint8_t t0 = a[0], t1 = a[1], ty = a[2];
    a += 3;
    if (t0 == 'R' && t1 == 'G') {
      if (ty != 'Z') return n_ids;
      const uint8_t* z = memchr(a, 0, (size_t)(end - a));
      if (!z) return n_ids;
      for (uint32_t g = 0; g < n_ids; ++g)
        if (strlen(ids[g]) == (size_t)(z - a) && !memcmp(ids[g], a, (size_t)(z - a))) return g;
      return n_ids;
    }
    size_t sz;
    switch (ty) {
      case 'A': case 'c': case 'C': sz = 1; break;
      case 's': case 'S': sz = 2; break;
      case 'i': case 'I': case 'f': sz = 4; break;
      case 'Z': case 'H': {
        const uint8_t* z = memchr(a, 0, (size_t)(end - a));
        if (!z) { snprintf(g_err, sizeof g_err, "aux %c%c:%c without NUL", t0, t1, ty); return -1; }
        sz = (size_t)(z - a) + 1;
        break;
      }
      case 'B': {
        if (end - a < 5) { snprintf(g_err, sizeof g_err, "aux B array header runs past the record"); return -1; }
        uint32_t cnt; memcpy(&cnt, a + 1, 4);
        size_t es = strchr("cC", a[0]) && a[0] ? 1 : strchr("sS", a[0]) && a[0] ? 2 : strchr("iIf", a[0]) && a[0] ? 4 : 0;
        if (!es) { snprintf(g_err, sizeof g_err, "aux B array of subtype %u", a[0]); return -1; }
        sz = 5 + (size_t)cnt * es;
        break;
      }
      default: snprintf(g_err, sizeof g_err, "aux field of type %u", ty); return -1;
    }
    if ((size_t)(end - a) < sz) { snprintf(g_err, sizeof g_err, "aux field runs past the record"); return -1; }
    a += sz;
  }
  return n_ids;
}

/* group: -1 = every record, 0..n_ids-1 = that read group, n_ids = the ungrouped records */
void* oracle_rg_run(const uint8_t* bam, size_t bam_len, uint64_t n_records, uint64_t gc_seed, const char* const* ids, uint32_t n_ids, int64_t group) {
  g_err[0] = 0;
  results_t* R = malloc(sizeof *R);
  results_init(R);
  R->do_records = 1;
  bgzf_t* rd = malloc(sizeof *rd);
  recbuf_t rb = {malloc(1 << 16), 1 << 16};
  rec_t rec;
  bgzf_open(rd, bam, bam_len);
  if (read_header(rd, &R->refs, &R->n_ref)) return NULL;
  uint64_t counter = 0;
  int rc;
  for (;;) {
    const uint64_t before = rg_stream_pos(rd);
    if ((rc = read_record(rd, &rb, &rec, R->n_ref)) != 1) break;
    const uint8_t* end = rb.buf + (rg_stream_pos(rd) - before - 4);
    const uint8_t* aux = rec.qual + rec.l_seq;
    const int64_t g = rg_group(aux, end, ids, n_ids);
    if (g < 0) return NULL;
    if (group < 0 || g == group) {
      if (general_process(R, &rec)) return NULL;
      tlen_process(R, &rec);
      gc_process(R, &rec, gc_seed);
      if (quality_process(R, &rec)) return NULL;
    }
    ++counter;
    if (n_records && counter >= n_records) break;
  }
  if (rc < 0) return NULL;
  R->pass1_records = counter;
  free(rd);
  free(rb.buf);
  return R;
}
