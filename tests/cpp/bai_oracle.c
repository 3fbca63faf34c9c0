/* bai_oracle.c — CPU restatement of the reference's `ngs index` for BAM (src/index/bam.rs:39-109): the checker the GPU BAI
 * build (NGSQ_F_INDEX, ngs_b200/csrc/index.cuh) is compared with.
 *
 * TEST INFRASTRUCTURE ONLY, like oracle/ngsqc_oracle.c, whose BGZF reader (noodles-bgzf restatement: CRC + ISIZE checks,
 * empty blocks skipped, own-address virtual offsets) and record decoder (read_header / read_record) it reuses by including
 * that file unchanged.  tests/baiutil.py compiles it on first use into a temporary directory:
 *   gcc -O2 -fPIC -shared -o libbai_oracle.so tests/cpp/bai_oracle.c -lz -lm
 * Entry points: oracle_build_bai (the .bai bytes), oracle_bai_keys (per-record keys); errors through oracle_last_error. */
#include "../../oracle/ngsqc_oracle.c"

/* ------------------------------------------------------------ BAI build (SURVEY 8(f) rank 4: `ngs index`)
 * Restates the indexing loop of src/index/bam.rs:39-109: the header is read (bam.rs:60-64), then every record, in file
 * order, goes to the indexer's add_record(alignment context, chunk) with the chunk running from the reader position before
 * the record to the position after it (bam.rs:74-96), and the index, built for the header's reference count
 * (bam.rs:98-100), is written as a .bai (bam.rs:102-107).  The rules below (key, chunks, linear index, order, limits) are
 * DESIGN.md section 4 (K13); the noodles behaviours they recall are SURVEY App. D.12.  Positions are own-address virtual
 * offsets (block of a record's first byte | offset in it), as read_record reports them (SURVEY F5 lists the deviation). */
typedef struct { int32_t ref, pos; uint32_t bin; uint64_t beg, end; int placed, unmapped; } bai_key_t;
static uint32_t bai_reg2bin(uint64_t beg, uint64_t end) { /* SAM spec 5.3 */
  --end;
  if (beg >> 14 == end >> 14) return ((1u << 15) - 1) / 7 + (uint32_t)(beg >> 14);
  if (beg >> 17 == end >> 17) return ((1u << 12) - 1) / 7 + (uint32_t)(beg >> 17);
  if (beg >> 20 == end >> 20) return ((1u << 9) - 1) / 7 + (uint32_t)(beg >> 20);
  if (beg >> 23 == end >> 23) return ((1u << 6) - 1) / 7 + (uint32_t)(beg >> 23);
  if (beg >> 26 == end >> 26) return ((1u << 3) - 1) / 7 + (uint32_t)(beg >> 26);
  return 0;
}
/* placed = ref >= 0 and pos >= 0: [pos, pos + span), a zero span counted as 1 (SAM spec; noodles: recalled, App. D.12) */
static int bai_key(const rec_t* r, bai_key_t* k) {
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
  if (k->end > (1ull << 29)) FAIL("record at virtual offset %llu ends at %llu: beyond what a BAI addresses (2^29)", (unsigned long long)r->voff, (unsigned long long)k->end);
  k->bin = bai_reg2bin(k->beg, k->end);
  return 0;
}
/* per record, in file order: ref, pos, bin, beg, end, placed, unmapped, virtual offset (8 int64); stops at the first record
 * the reader or the indexer rejects (returns -1; the records before it are written) */
int oracle_bai_keys(const uint8_t* bam, size_t bam_len, int64_t* out, size_t cap, size_t* n_out) {
  g_err[0] = 0; *n_out = 0;
  bgzf_t* rd = malloc(sizeof *rd); recbuf_t rb = {malloc(1 << 16), 1 << 16}; rec_t rec; ref_t* refs; uint32_t n_ref;
  bgzf_open(rd, bam, bam_len);
  int ret = read_header(rd, &refs, &n_ref);
  size_t n = 0; int rc;
  while (!ret && (rc = read_record(rd, &rb, &rec, n_ref)) == 1) {
    bai_key_t k;
    if (bai_key(&rec, &k)) { ret = -1; break; }
    if (n < cap) { int64_t* o = out + 8 * n; o[0] = k.ref; o[1] = k.pos; o[2] = k.bin; o[3] = (int64_t)k.beg; o[4] = (int64_t)k.end; o[5] = k.placed; o[6] = k.unmapped; o[7] = (int64_t)rec.voff; }
    ++n;
  }
  if (!ret && rc < 0) ret = -1;
  *n_out = n; free(rd); free(rb.buf);
  return ret;
}

typedef struct { uint32_t bin, n, cap; chunk_t* v; } bbin_t;
typedef struct { bbin_t* bins; uint32_t n_bins, cap_bins; uint64_t beg, end, n_mapped, n_unmapped; int any; uint64_t* lin; uint32_t n_lin; } bref_t;
typedef struct { uint8_t* p; size_t n, cap; } bbuf_t;
static void bput(bbuf_t* b, const void* v, size_t k) { if (b->n + k > b->cap) { b->cap = (b->n + k) * 2; b->p = realloc(b->p, b->cap); } memcpy(b->p + b->n, v, k); b->n += k; }
static void bput32(bbuf_t* b, uint32_t v) { bput(b, &v, 4); }
static void bput64(bbuf_t* b, uint64_t v) { bput(b, &v, 8); }
/* closes a run of records with one (ref, bin): a chunk of that bin, merged into the bin's last chunk when contiguous */
static void bai_close_run(bref_t* R, uint32_t bin, uint64_t beg, uint64_t end) {
  bbin_t* B = NULL;
  for (uint32_t i = 0; i < R->n_bins; ++i) if (R->bins[i].bin == bin) { B = &R->bins[i]; break; }
  if (!B) { /* bins in order of first use */
    if (R->n_bins == R->cap_bins) { R->cap_bins = R->cap_bins ? 2 * R->cap_bins : 16; R->bins = realloc(R->bins, R->cap_bins * sizeof *R->bins); }
    B = &R->bins[R->n_bins++]; memset(B, 0, sizeof *B); B->bin = bin;
  }
  if (B->n && B->v[B->n - 1].end == beg) { B->v[B->n - 1].end = end; }
  else { if (B->n == B->cap) { B->cap = B->cap ? 2 * B->cap : 4; B->v = realloc(B->v, B->cap * sizeof *B->v); } B->v[B->n].beg = beg; B->v[B->n].end = end; B->n++; }
  if (!R->any) { R->any = 1; R->beg = beg; }
  R->end = end;
}
/* The .bai of `bam` into out[0, cap) (when it fits); *n_out = its size.  0, or -1 with oracle_last_error() (a record the
 * reader rejects, a record beyond 2^29, unsorted records). */
int oracle_build_bai(const uint8_t* bam, size_t bam_len, uint8_t* out, size_t cap, size_t* n_out) {
  g_err[0] = 0; *n_out = 0;
  bgzf_t* rd = malloc(sizeof *rd); recbuf_t rb = {malloc(1 << 16), 1 << 16}; rec_t rec; ref_t* refs; uint32_t n_ref;
  bgzf_open(rd, bam, bam_len);
  if (read_header(rd, &refs, &n_ref)) return -1;
  bref_t* R = calloc(n_ref ? n_ref : 1, sizeof *R);
  uint64_t n_no_coor = 0;
  /* the open run: key (ref, bin) or none / unplaced, and its first offset */
  int run_open = 0, run_placed = 0; int32_t run_ref = -1; uint32_t run_bin = 0; uint64_t run_beg = 0;
  /* order: the last record that constrains it (placed, or ref = -1) */
  int have_last = 0, seen_no_ref = 0; int32_t last_ref = 0, last_pos = 0;
  uint64_t end_data;
  for (;;) {
    uint64_t before = bgzf_tell(rd); /* the position after the previous record when this read finds EOF */
    int rc = read_record(rd, &rb, &rec, n_ref);
    if (rc < 0) return -1;
    if (rc == 0) { end_data = before; break; }
    bai_key_t k;
    if (bai_key(&rec, &k)) return -1;
    const uint64_t v = rec.voff;
    if (k.placed) {
      if (seen_no_ref || (have_last && (k.ref < last_ref || (k.ref == last_ref && k.pos < last_pos))))
        FAIL("unsorted records: the record at virtual offset %llu is out of coordinate order", (unsigned long long)v);
      have_last = 1; last_ref = k.ref; last_pos = k.pos;
    } else if (k.ref < 0) seen_no_ref = 1;
    /* a record whose key differs from the open run's ends that run here (an unplaced record ends a run, joins none) */
    if (run_open && !(k.placed && run_placed && k.ref == run_ref && k.bin == run_bin)) {
      if (run_placed) bai_close_run(&R[run_ref], run_bin, run_beg, v);
      run_open = 0;
    }
    if (!k.placed) { n_no_coor++; continue; }
    if (!run_open) { run_open = 1; run_placed = 1; run_ref = k.ref; run_bin = k.bin; run_beg = v; }
    bref_t* F = &R[k.ref];
    if (k.unmapped) F->n_unmapped++; else F->n_mapped++;
    /* linear index: window w keeps the offset of the first record touching it (~0 = none yet) */
    uint32_t w0 = (uint32_t)(k.beg >> 14), w1 = (uint32_t)((k.end - 1) >> 14);
    if (w1 + 1 > F->n_lin) { F->lin = realloc(F->lin, (w1 + 1) * 8ull); for (uint32_t w = F->n_lin; w <= w1; ++w) F->lin[w] = ~0ull; F->n_lin = w1 + 1; }
    for (uint32_t w = w0; w <= w1; ++w) if (F->lin[w] == ~0ull) F->lin[w] = v;
  }
  if (run_open && run_placed) bai_close_run(&R[run_ref], run_bin, run_beg, end_data);
  bbuf_t b = {NULL, 0, 0};
  bput(&b, "BAI\1", 4); bput32(&b, n_ref);
  for (uint32_t c = 0; c < n_ref; ++c) {
    bref_t* F = &R[c];
    if (!F->any) { bput32(&b, 0); bput32(&b, 0); continue; }
    bput32(&b, F->n_bins + 1);
    for (uint32_t i = 0; i < F->n_bins; ++i) {
      bput32(&b, F->bins[i].bin); bput32(&b, F->bins[i].n);
      for (uint32_t j = 0; j < F->bins[i].n; ++j) { bput64(&b, F->bins[i].v[j].beg); bput64(&b, F->bins[i].v[j].end); }
      free(F->bins[i].v);
    }
    bput32(&b, 37450); bput32(&b, 2); bput64(&b, F->beg); bput64(&b, F->end); bput64(&b, F->n_mapped); bput64(&b, F->n_unmapped);
    /* windows no record touched take the previous window's value (0 before the first touched one) */
    uint64_t last = 0;
    bput32(&b, F->n_lin);
    for (uint32_t w = 0; w < F->n_lin; ++w) { if (F->lin[w] != ~0ull) last = F->lin[w]; bput64(&b, last); }
    free(F->bins); free(F->lin);
  }
  bput64(&b, n_no_coor);
  *n_out = b.n;
  if (out && cap >= b.n) memcpy(out, b.p, b.n);
  free(b.p); free(R); free(rd); free(rb.buf);
  return 0;
}

