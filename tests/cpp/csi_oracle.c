/* csi_oracle.c — CPU restatement of `samtools index -c` for BAM: the checker the GPU CSI build (NGSQ_F_INDEX_CSI,
 * ngs_b200/csrc/index.cuh) is compared with.
 *
 * TEST INFRASTRUCTURE ONLY.  It includes the BAI oracle (tests/cpp/bai_oracle.c) unchanged, and with it the BGZF reader and
 * record decoder of oracle/ngsqc_oracle.c, and restates the BAI's indexing loop at a CSI binning.  tests/csiutil.py compiles
 * it on first use into a temporary directory:
 *   gcc -O2 -fPIC -shared -o libcsi_oracle.so tests/cpp/csi_oracle.c -lz -lm
 * Entry points: oracle_build_csi (the uncompressed .csi payload), oracle_csi_keys (per-record keys), oracle_csi_default_depth;
 * errors through oracle_last_error. */
#include "bai_oracle.c"

/* ------------------------------------------------------------ CSI build (`samtools index -c`; DESIGN.md section 4, "K13 CSI")
 * The same loop as oracle_build_bai, at the binning (min_shift, depth) of CSIv1: bins are hts_reg2bin(beg, end, min_shift,
 * depth), records may end at most at 2^(min_shift + 3 depth), the windows are 2^min_shift bases wide, and every bin carries
 * loffset = the filled window minimum at its first leaf window (hts_bin_bot; 0 past the last touched window, and untouched
 * windows before the first touched one hold 0, as in the BAI).  depth = 0: the smallest n with max_len + 256 <= 2^(min_shift +
 * 3n) over the header's lengths.  The payload is returned uncompressed. */
static uint32_t csi_reg2bin(uint64_t beg, uint64_t end, int min_shift, int depth) { /* htslib hts_reg2bin (CSIv1) */
  int l, s = min_shift; uint32_t t = ((1u << (3 * depth)) - 1) / 7;
  for (--end, l = depth; l > 0; --l, s += 3, t -= 1u << (3 * l))
    if (beg >> s == end >> s) return t + (uint32_t)(beg >> s);
  return 0;
}
static uint64_t csi_bin_bot(uint32_t bin, int depth) { /* htslib hts_bin_bot */
  int l = 0;
  for (uint32_t b = bin; b; b = (b - 1) >> 3) ++l;
  return (uint64_t)(bin - ((1u << (3 * l)) - 1) / 7) << (3 * (depth - l));
}
int oracle_csi_default_depth(uint64_t max_len, int min_shift) {
  int n = 0;
  for (uint64_t s = 1ull << min_shift; max_len + 256 > s; s <<= 3) ++n;
  return n;
}
static int csi_key(const rec_t* r, int min_shift, int depth, bai_key_t* k) {
  k->ref = r->ref_id; k->pos = r->pos; k->placed = r->ref_id >= 0 && r->pos >= 0; k->unmapped = (r->flag & 4) != 0;
  k->bin = 0; k->beg = k->end = 0;
  if (!k->placed) return 0;
  uint64_t span = 0;
  for (uint32_t i = 0; i < r->n_cigar; ++i) {
    uint32_t op; memcpy(&op, (const uint8_t*)r->cigar + 4 * i, 4);
    uint32_t kind = op & 15;
    if (kind == 0 || kind == 2 || kind == 3 || kind == 7 || kind == 8) span += op >> 4;
  }
  k->beg = (uint64_t)r->pos; k->end = k->beg + (span ? span : 1);
  if (k->end > (1ull << (min_shift + 3 * depth)))
    FAIL("record at virtual offset %llu ends at %llu: beyond what a CSI of min_shift %d and depth %d addresses (2^%d)", (unsigned long long)r->voff,
         (unsigned long long)k->end, min_shift, depth, min_shift + 3 * depth);
  k->bin = csi_reg2bin(k->beg, k->end, min_shift, depth);
  return 0;
}
static int csi_depth_of(const ref_t* refs, uint32_t n_ref, int min_shift, int depth) {
  if (depth) return depth;
  uint64_t mx = 0;
  for (uint32_t c = 0; c < n_ref; ++c) if (refs[c].len > mx) mx = refs[c].len;
  return oracle_csi_default_depth(mx, min_shift);
}
/* oracle_bai_keys at a CSI binning (depth 0: the default rule); *depth_out = the depth used */
int oracle_csi_keys(const uint8_t* bam, size_t bam_len, int min_shift, int depth, int64_t* out, size_t cap, size_t* n_out, int* depth_out) {
  g_err[0] = 0; *n_out = 0;
  bgzf_t* rd = malloc(sizeof *rd); recbuf_t rb = {malloc(1 << 16), 1 << 16}; rec_t rec; ref_t* refs; uint32_t n_ref;
  bgzf_open(rd, bam, bam_len);
  int ret = read_header(rd, &refs, &n_ref);
  if (!ret) depth = csi_depth_of(refs, n_ref, min_shift, depth);
  *depth_out = depth;
  size_t n = 0; int rc;
  while (!ret && (rc = read_record(rd, &rb, &rec, n_ref)) == 1) {
    bai_key_t k;
    if (csi_key(&rec, min_shift, depth, &k)) { ret = -1; break; }
    if (n < cap) { int64_t* o = out + 8 * n; o[0] = k.ref; o[1] = k.pos; o[2] = k.bin; o[3] = (int64_t)k.beg; o[4] = (int64_t)k.end; o[5] = k.placed; o[6] = k.unmapped; o[7] = (int64_t)rec.voff; }
    ++n;
  }
  if (!ret && rc < 0) ret = -1;
  *n_out = n; free(rd); free(rb.buf);
  return ret;
}
/* The .csi payload of `bam` at (min_shift, depth; 0 = the default rule) into out[0, cap) (when it fits); *n_out = its size.
 * 0, or -1 with oracle_last_error() (a record the reader rejects, a record past 2^(min_shift + 3 depth), a reference longer
 * than that, unsorted records). */
int oracle_build_csi(const uint8_t* bam, size_t bam_len, int min_shift, int depth, uint8_t* out, size_t cap, size_t* n_out) {
  g_err[0] = 0; *n_out = 0;
  bgzf_t* rd = malloc(sizeof *rd); recbuf_t rb = {malloc(1 << 16), 1 << 16}; rec_t rec; ref_t* refs; uint32_t n_ref;
  bgzf_open(rd, bam, bam_len);
  if (read_header(rd, &refs, &n_ref)) return -1;
  depth = csi_depth_of(refs, n_ref, min_shift, depth);
  for (uint32_t c = 0; c < n_ref; ++c)
    if ((uint64_t)refs[c].len > (1ull << (min_shift + 3 * depth))) FAIL("reference %u is longer than a CSI of min_shift %d and depth %d addresses", c, min_shift, depth);
  bref_t* R = calloc(n_ref ? n_ref : 1, sizeof *R);
  uint64_t n_no_coor = 0;
  int run_open = 0, run_placed = 0; int32_t run_ref = -1; uint32_t run_bin = 0; uint64_t run_beg = 0;
  int have_last = 0, seen_no_ref = 0; int32_t last_ref = 0, last_pos = 0;
  uint64_t end_data;
  for (;;) {
    uint64_t before = bgzf_tell(rd);
    int rc = read_record(rd, &rb, &rec, n_ref);
    if (rc < 0) return -1;
    if (rc == 0) { end_data = before; break; }
    bai_key_t k;
    if (csi_key(&rec, min_shift, depth, &k)) return -1;
    const uint64_t v = rec.voff;
    if (k.placed) {
      if (seen_no_ref || (have_last && (k.ref < last_ref || (k.ref == last_ref && k.pos < last_pos))))
        FAIL("unsorted records: the record at virtual offset %llu is out of coordinate order", (unsigned long long)v);
      have_last = 1; last_ref = k.ref; last_pos = k.pos;
    } else if (k.ref < 0) seen_no_ref = 1;
    if (run_open && !(k.placed && run_placed && k.ref == run_ref && k.bin == run_bin)) {
      if (run_placed) bai_close_run(&R[run_ref], run_bin, run_beg, v);
      run_open = 0;
    }
    if (!k.placed) { n_no_coor++; continue; }
    if (!run_open) { run_open = 1; run_placed = 1; run_ref = k.ref; run_bin = k.bin; run_beg = v; }
    bref_t* F = &R[k.ref];
    if (k.unmapped) F->n_unmapped++; else F->n_mapped++;
    uint32_t w0 = (uint32_t)(k.beg >> min_shift), w1 = (uint32_t)((k.end - 1) >> min_shift);
    if (w1 + 1 > F->n_lin) { F->lin = realloc(F->lin, (w1 + 1) * 8ull); for (uint32_t w = F->n_lin; w <= w1; ++w) F->lin[w] = ~0ull; F->n_lin = w1 + 1; }
    for (uint32_t w = w0; w <= w1; ++w) if (F->lin[w] == ~0ull) F->lin[w] = v;
  }
  if (run_open && run_placed) bai_close_run(&R[run_ref], run_bin, run_beg, end_data);
  const uint32_t n_bins = ((1u << (3 * (depth + 1))) - 1) / 7;
  bbuf_t b = {NULL, 0, 0};
  bput(&b, "CSI\1", 4); bput32(&b, (uint32_t)min_shift); bput32(&b, (uint32_t)depth); bput32(&b, 0); bput32(&b, n_ref);
  for (uint32_t c = 0; c < n_ref; ++c) {
    bref_t* F = &R[c];
    if (!F->any) { bput32(&b, 0); continue; }
    uint64_t last = 0; /* fill: untouched windows take the previous window's value (0 before the first touched one) */
    for (uint32_t w = 0; w < F->n_lin; ++w) { if (F->lin[w] != ~0ull) last = F->lin[w]; F->lin[w] = last; }
    bput32(&b, F->n_bins + 1);
    for (uint32_t i = 0; i < F->n_bins; ++i) {
      const uint64_t bot = csi_bin_bot(F->bins[i].bin, depth);
      bput32(&b, F->bins[i].bin); bput64(&b, bot < F->n_lin ? F->lin[bot] : 0); bput32(&b, F->bins[i].n);
      for (uint32_t j = 0; j < F->bins[i].n; ++j) { bput64(&b, F->bins[i].v[j].beg); bput64(&b, F->bins[i].v[j].end); }
      free(F->bins[i].v);
    }
    bput32(&b, n_bins + 1); bput64(&b, 0); bput32(&b, 2); bput64(&b, F->beg); bput64(&b, F->end); bput64(&b, F->n_mapped); bput64(&b, F->n_unmapped);
    free(F->bins); free(F->lin);
  }
  bput64(&b, n_no_coor);
  *n_out = b.n;
  if (out && cap >= b.n) memcpy(out, b.p, b.n);
  free(b.p); free(R); free(rd); free(rb.buf);
  return 0;
}
