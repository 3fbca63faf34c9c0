/* ngs_cuda.h — C ABI of libngs_cuda.so, the B200 engine behind `ngs qc`.
 *
 * This is the drop-in boundary for the reference's BAM quality-control hot path
 * (stjude-rust-labs/ngs v0.4.0).  A Rust `ngs-cuda` module binds exactly these
 * symbols (see INTEGRATION.md for the `extern "C"` block and the `app()` branch);
 * in this repository the same symbols are driven by the C++ host driver
 * (ngs_b200/host) and by ctypes (ngs_b200/ffi.py).
 *
 * What each entry point replaces on the reference side:
 *   ngsq_submit*            BGZF read + inflate + CRC/ISIZE check done by
 *                           bam::Reader / noodles-bgzf (src/utils/formats/bam.rs:41-44,
 *                           src/qc/command.rs:305 and :350 — the reference inflates twice).
 *   ngsq_finish             the two hot loops of app(): src/qc/command.rs:305-316 (pass 1,
 *                           every record through every record-based facet) and :350-397
 *                           (pass 2, per-contig query -> Coverage.process/teardown), i.e.
 *                           the process() bodies of general.rs:31-124, template_length.rs:79-87,
 *                           gc_content.rs:38-100, quality_scores.rs:37-49, coverage.rs:148-262.
 *   ngsq_get_*              the integer state those facets hold when summarize()/aggregate()
 *                           run (general/metrics.rs:10-136, template_length.rs:14-53,
 *                           gc_content/metrics.rs:10-68, quality_scores.rs:16-19,
 *                           coverage.rs:28-69).  The engine returns INTEGERS ONLY; every derived
 *                           float is computed by the caller in the reference's operation order.
 *   ngsq_reduce             nothing (the reference is single-process); merges shards.
 *
 * Conventions: plain pointers and sizes, caller owns every in/out buffer, no callbacks, no
 * memory returned that the caller must free.  Every function returns NGSQ_OK or a negative
 * NGSQ_E_* code; ngsq_last_error() gives the message.  An engine handle is not thread-safe:
 * one handle per GPU, one host thread per handle.  There is no CPU fallback: without a CUDA
 * device ngsq_create fails with NGSQ_E_CUDA.
 */
#ifndef NGS_CUDA_H_
#define NGS_CUDA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NGSQ_VERSION 0x000100

enum {
  NGSQ_OK = 0,
  NGSQ_E_ARG = -1,        /* bad argument / call order */
  NGSQ_E_CUDA = -2,       /* CUDA runtime failure (message has the CUDA error) */
  NGSQ_E_TRUNCATED = -3,  /* BGZF data ends inside a block / record chain runs past the data */
  NGSQ_E_BAD_BLOCK = -4,  /* malformed BGZF framing or DEFLATE stream, ISIZE mismatch */
  NGSQ_E_CRC = -5,        /* CRC32 of an inflated block does not match its trailer */
  NGSQ_E_BAD_RECORD = -6, /* malformed BAM record (op > 8, refID >= n_ref, fields overrun ...) */
  NGSQ_E_QUAL_RANGE = -7, /* quality score > 93 (the reference's decoder aborts the run) */
  NGSQ_E_CHAIN = -8,      /* record-boundary closure check failed */
  NGSQ_E_NCCL = -9,
  NGSQ_E_NOMEM = -10,
  NGSQ_E_EDITS = -11,     /* the Edits facet met a record / reference the reference program aborts on */
  NGSQ_E_FEATURES = -12,  /* likewise for the Genomic Features facet */
  NGSQ_E_QUAL_CAP = -13,  /* a read is longer than the quality table: raise quality_positions and run again */
  NGSQ_E_UNSORTED = -14   /* NGSQ_F_INDEX: the records are not coordinate-sorted (the message names the first offender) */
};

/* ngsq_config.flags */
#define NGSQ_F_RECORD_FACETS 1u /* General, Template Length, GC Content, Quality Score */
#define NGSQ_F_COVERAGE 2u      /* Coverage */
#define NGSQ_F_VERIFY_CRC 4u    /* verify the CRC32 of every block (reference behaviour) */
#define NGSQ_F_EDITS 8u         /* Edits (needs ngsq_set_reference_bases for every contig that holds records) */
#define NGSQ_F_FEATURES 16u     /* Genomic Features (needs ngsq_set_feature_model + ngsq_set_features) */
#define NGSQ_F_SERIAL_STAGES 32u /* measurement aid: every kernel of a wave on ONE stream (no overlap with the next wave's
                                    inflate), so that per-stage event times are the kernels' own; results are identical */
#define NGSQ_F_INDEX 64u        /* build the file's BAI in the same pass (`ngs index`, src/index/bam.rs:39-109); combines with every
                                   other flag.  The range must start at the first record and reach to the end (end_voffset 0),
                                   max_records must be 0, references must be shorter than 2^29 (longer ones need CSI) and the
                                   records coordinate-sorted (NGSQ_E_UNSORTED otherwise).  Read the bytes with ngsq_get_bai. */
#define NGSQ_F_INDEX_PART 128u  /* index ONE contiguous range of a file cut between engines; set instead of NGSQ_F_INDEX (both:
                                   NGSQ_E_ARG), combines with every other flag.  The range is [first, end) of ngsq_set_range (end 0 =
                                   to the end of the data); max_records must be 0; ngsq_reduce and the split-reference calls are
                                   allowed.  ngsq_finish keeps the part's index state on the host without assembling it, and does not
                                   check the order (it is checked across the parts by the join); ngsq_get_bai is refused: join the
                                   finished parts with ngsq_join_bai. */
#define NGSQ_F_INDEX_CSI 256u  /* with NGSQ_F_INDEX or NGSQ_F_INDEX_PART: build a CSI instead of a BAI (alone: NGSQ_E_ARG).  Bins are
                                   CSIv1's hts_reg2bin(beg, end, min_shift, depth) (ngsq_set_index_binning; default min_shift 14 and
                                   samtools' depth rule), records may end at most at 2^(min_shift + 3 depth) and references may be at
                                   most that long.  Read the bytes with ngsq_get_csi, join parts with ngsq_join_csi. */
#define NGSQ_F_READ_GROUPS 512u  /* with NGSQ_F_RECORD_FACETS (alone: NGSQ_E_ARG): the four record facets once more per read group
                                    (ngsq_set_read_groups, ngsq_select_read_group); the sample's results are unchanged */

typedef struct ngsq_engine ngsq_engine;

typedef struct ngsq_config {
  uint32_t struct_size;        /* sizeof(ngsq_config) */
  uint32_t flags;              /* NGSQ_F_* */
  uint64_t gc_seed;            /* GC window policy: see ngsq_get_gc */
  uint64_t max_records;        /* `-n` (command.rs:305-316 and :384-388): pass 1 takes the first N records in file order;
                                  pass 2 (Coverage) applies the reference's shared counter: the first N records its
                                  per-contig queries yield, then the first yielded record of every later contig; 0 = all */
  uint64_t reserve_compressed; /* optional: size of the whole compressed shard.  Set -> it stays resident in one device
                                  buffer; 0 -> a staging ring of comp_ring_bytes that is recycled wave by wave */
  uint64_t reserve_inflated;   /* optional: inflated size of the shard (sizes the two wave slots once) */
  uint32_t reserve_blocks;     /* optional: BGZF blocks of the shard (equal waves, a small last wave) */
  uint32_t launch_blocks;      /* tuning/testing: BGZF blocks per wave; 0 = one block per lane of the decode kernel
                                  (SMs x 576 lanes) */
  uint32_t quality_positions;  /* rows of the quality-by-position table = longest read the run may hold; 0 = 131072 */
  uint32_t carry_bytes;        /* longest record that may straddle two waves; 0 = 16 MiB */
  uint64_t comp_ring_bytes;    /* device bytes of the compressed staging ring when reserve_compressed is 0; 0 = 8 GiB */
} ngsq_config;

/* One BGZF block as framed by the host (K1). */
typedef struct ngsq_block {
  uint64_t coffset;  /* file offset of the block's first byte (gzip magic) */
  uint32_t hdr_len;  /* bytes before the DEFLATE payload (12 + XLEN) */
  uint32_t csize;    /* total block size (BSIZE + 1) */
  uint32_t isize;    /* inflated size from the trailer */
  uint32_t crc32;    /* CRC32 from the trailer */
} ngsq_block;

typedef struct ngsq_stats {
  uint64_t records;          /* records owned by this shard (all, before `-n`) */
  uint64_t blocks;           /* BGZF blocks submitted (non-empty) */
  uint64_t compressed_bytes; /* BGZF bytes submitted */
  uint64_t inflated_bytes;   /* sum of ISIZE */
  uint64_t max_read_len;     /* longest l_seq seen */
  /* Stage times are sums over the waves of CUDA-event intervals on the stage's own stream.  The scan / facet / CRC kernels of
   * wave k run beside the inflate of wave k+1, so the stages overlap (their sum exceeds ms_total) and each includes the time
   * it shared the SMs with the others; NGSQ_F_SERIAL_STAGES gives the kernels' own times. */
  float ms_inflate;          /* device time of the inflate launches (bitmap clear + decode + resolve; CUDA events) */
  float ms_crc;
  float ms_scan;             /* record-boundary discovery + offset table */
  float ms_facets;           /* fused record-facet + coverage-scatter kernel, and the other per-wave record kernels (Edits,
                                Genomic Features, the NGSQ_F_INDEX key / run kernel, the NGSQ_F_READ_GROUPS kernels) */
  float ms_coverage;         /* difference-array resolve */
  float ms_total;            /* first submit -> end of finish on the engine's stream */
  uint32_t inflate_launches, other_launches;
  float ms_inflate_decode;   /* of ms_inflate: the lane-per-block Huffman decode kernel */
  float ms_inflate_resolve;  /* of ms_inflate: the warp-per-block LZ77 resolve kernel */
  float ms_reduce;           /* ngsq_reduce: agreement all-reduce + split-reference reduce and resolve + sum-reduce + refresh
                                (0 without it) */
  float ms_edits;            /* VAF histogram of the Edits facet (its per-record kernel runs inside ms_facets) */
  float ms_tail;             /* start of the LAST wave -> end of finish: what is left once the last chunk has arrived */
  uint32_t waves;            /* inflate waves of the run (= inflate_launches) */
} ngsq_stats;

int ngsq_version(void);
const char* ngsq_last_error(ngsq_engine* e); /* e may be NULL: error of the failed ngsq_create */

int ngsq_create(int device, const ngsq_config* cfg, ngsq_engine** out);
void ngsq_destroy(ngsq_engine* e);
/* Forget all submitted data and zero every accumulator; allocations and references are kept. */
int ngsq_reset(ngsq_engine* e);

/* Reference sequences from the BAM header (lengths) and, per reference, whether Coverage
 * processes it (CoverageFacet::supports_sequence_name, coverage.rs:133-138 — decided by the
 * caller from the genome's primary-assembly table).  Must precede the first submit. */
int ngsq_set_references(ngsq_engine* e, uint32_t n_ref, const uint32_t* ref_len, const uint8_t* coverage_enabled);

/* Edits facet (src/qc/sequence_based/edits.rs:175-215, setup): the letters of reference `ref`'s sequence from the
 * reference FASTA, line ends removed, as they stand in the file (the engine applies noodles' Base::try_from rule:
 * the sixteen upper-case letters "=ACMGRSVTWYHKDBN"; a record over any other letter fails the run as it does in the
 * reference).  After ngsq_set_references, before the first submit; the caller reports "sequence not found" itself
 * for contigs the FASTA lacks (a record on a contig without a sequence fails the run).  Needs NGSQ_F_EDITS. */
int ngsq_set_reference_bases(ngsq_engine* e, uint32_t ref, const uint8_t* letters, uint64_t n);

/* Genomic Features facet (src/qc/record_based/features.rs:270-355, try_from): the gene model, filed the way the
 * reference files it.  The five configured feature names are slots 0 five_prime_utr, 1 three_prime_utr,
 * 2 coding_sequence, 3 exon, 4 gene (command.rs:78-101); names may coincide, so slot_class[j] = the smallest slot index
 * whose name equals slot j's.  primary[c] = reference c is in the genome's primary assembly (features.rs:157-164).
 * Then, per primary reference, every GFF record whose type equals one of the names: start, end (1-based, as they stand
 * in the GFF; end is used as an exclusive bound like the reference does) and cls = slot_class of the FIRST slot whose
 * name equals the type.  GFF parsing, the strand check of features/utils.rs:33-43 and "unwrap every record" stay on the
 * caller's side.  After ngsq_set_references, before the first submit.  Needs NGSQ_F_FEATURES. */
int ngsq_set_feature_model(ngsq_engine* e, const uint8_t slot_class[5], const uint8_t* primary);
int ngsq_set_features(ngsq_engine* e, uint32_t ref, uint32_t n, const uint32_t* start, const uint32_t* stop, const uint8_t* cls);

/* Virtual offsets (coffset << 16 | uoffset) of the first record this shard owns and of the
 * first record it does NOT own (0 = everything to the end of the submitted data).  Both must
 * be true record starts (after the header for shard 0; BAI anchors otherwise). */
int ngsq_set_range(ngsq_engine* e, uint64_t first_rec_voffset, uint64_t end_voffset);

/* K1 helper: walks the BGZF chain in `bgzf` (file bytes starting at a block boundary at file
 * offset `file_off`).  Writes up to `cap` descriptors, *n_blocks = blocks found, *consumed =
 * bytes covered by whole blocks (a trailing partial block is not an error: resubmit it with
 * the next chunk). */
int ngsq_bgzf_walk(const uint8_t* bgzf, size_t nbytes, uint64_t file_off, ngsq_block* out, uint32_t cap,
                   uint32_t* n_blocks, size_t* consumed);

/* Streams one chunk of whole BGZF blocks from HOST memory: async H2D copy into the staging ring; a WAVE (inflate ->
 * CRC -> record scan -> facet kernels) is enqueued whenever launch_blocks blocks have been copied (and by ngsq_finish
 * for the rest), so the copy of one chunk overlaps the kernels of the previous ones and the device footprint does not
 * grow with the file.  The call never waits for the GPU unless the ring is full.  The buffer must stay valid until its
 * copy has completed (ngsq_wait_copied, or ngsq_finish).  Chunks must be submitted in file order; ngsq_set_range first. */
int ngsq_submit(ngsq_engine* e, const uint8_t* bgzf, size_t nbytes, uint64_t file_off);
/* Enqueues a wave for every block submitted so far instead of waiting for a full one.  A caller that knows its last
 * chunk calls this just before submitting it: what remains after the last copied byte is then one small wave. */
int ngsq_flush(ngsq_engine* e);
/* Several files in one run (`qc --cuda-also`, DESIGN.md section 5, "Several files"): the chunks submitted since the last
 * ngsq_set_range form one whole file.  This call enqueues that file's last wave as ngsq_flush does, so that no wave holds
 * blocks of two files, and a record still open at its end fails the run with NGSQ_E_TRUNCATED at ngsq_finish.  It drops the
 * open-record carry and the end-of-range state, so no record chain links two files, and leaves every accumulator as it is:
 * the facet histograms, Coverage's difference arrays and touched words, the Edits and Genomic Features state, the quality
 * table and the stats (ngsq_get_stats sums over the files of the run).  The caller then calls ngsq_set_range for the next
 * file and submits its chunks at that file's own offsets; ngsq_finish (and ngsq_reduce) run once, after the last file.  A
 * file may contribute nothing: ngsq_set_range, no submit, ngsq_next_file.  NGSQ_E_ARG after ngsq_finish, with NGSQ_F_INDEX or
 * NGSQ_F_INDEX_PART (an index describes one file), with max_records != 0 (`-n` counts in one file's order), and before the
 * file's ngsq_set_range.  The GC window of a record is keyed by its virtual offset in its own file. */
int ngsq_next_file(ngsq_engine* e);
/* Read groups (`qc --cuda-by-read-group`, DESIGN.md section 5, "Read groups"), with NGSQ_F_READ_GROUPS: the @RG IDs of the
 * header(s), `ids` = n NUL-terminated IDs back to back in ids_bytes bytes.  Group g < n is the records whose FIRST aux field
 * tagged RG (htslib's bam_aux_get) is of type Z and equals ID g byte for byte; group n ("ungrouped") is every other record:
 * no RG field, an RG field of another type, or a value no ID matches.  Records outside max_records belong to no group.  With
 * the flag, the aux fields in front of a record's first RG field are read, and a malformed one (unknown type, no NUL, a field
 * that runs past the record) fails the run with NGSQ_E_BAD_RECORD; without it aux bytes are never read.  Each of the n + 1
 * groups holds the integers of the four record facets: the 34 of ngsq_get_general, the TLEN histogram and its two counters,
 * the GC histogram with its nucleobase and record counters, and a quality length and table with as many rows as the sample's
 * (ngsq_set_quality_positions resizes both): (n + 1) x (1169 + 94 x rows) x 8 bytes of device memory in one buffer apart from
 * the packed result buffer (about 99 MB per group at the default 131072 rows).  A group's reads are never longer than the
 * sample's, so NGSQ_E_QUAL_CAP covers the group tables too.  After ngsq_set_references, before the first submit; kept across
 * ngsq_reset and ngsq_next_file accumulates like every other result.  NGSQ_E_ARG without the flag, for n > 65534, an empty or
 * repeated ID or ids_bytes that does not hold exactly n IDs; NGSQ_E_NOMEM (naming n and the rows) when the tables do not fit.
 * ngsq_reduce merges the groups too: the quality lengths with max, the rest with sum; the ranks must agree on n, the IDs and
 * the rows (NGSQ_E_ARG before any group data moves). */
int ngsq_set_read_groups(ngsq_engine* e, uint32_t n, const char* ids, size_t ids_bytes);
/* After ngsq_finish (and ngsq_reduce): which results the getters return.  -1 (the default, and again after ngsq_reset) is the
 * sample; 0..n a group (n = ungrouped).  While a group is selected, ngsq_get_general, ngsq_get_tlen, ngsq_get_gc and
 * ngsq_get_quality return that group's integers in the sample's layout, and the Coverage, Edits, Genomic Features and
 * edit-position getters fail with NGSQ_E_ARG (those facets are the sample's only).  NGSQ_E_ARG before ngsq_finish, without
 * NGSQ_F_READ_GROUPS, or for g outside [-1, n]. */
int ngsq_select_read_group(ngsq_engine* e, int32_t g);
/* Records whose wave has been scanned so far (never blocks; lags the submits by about one wave): the caller's
 * RecordCounter log line, src/utils/display.rs:43-52. */
int ngsq_progress(ngsq_engine* e, uint64_t* records);
/* Blocks until the host buffer of this run's submit_index-th ngsq_submit (0-based) has been copied to the device:
 * the caller may then refill it (pinned double-buffered file readers). */
int ngsq_wait_copied(ngsq_engine* e, uint32_t submit_index);
/* Same for a chunk already resident in DEVICE memory (used in place, not copied); the caller
 * passes the descriptors ngsq_bgzf_walk produced for it.  The allocation must stay readable for 64 bytes
 * past nbytes: the decoders read their input through aligned 8-byte windows that run ahead of the last
 * block's end (ngsq_submit pads its own copies). */
int ngsq_submit_device(ngsq_engine* e, const void* dev_bgzf, size_t nbytes, const ngsq_block* blocks, uint32_t n_blocks);

/* Last wave, coverage resolve, result read-back; blocks until the device is done. */
int ngsq_finish(ngsq_engine* e);

/* ---- integer results (valid after ngsq_finish / ngsq_reduce) ---- */
/* out[0..16): total, unmapped, duplicate, primary, secondary, supplementary, primary_mapped,
 * primary_duplicate, paired, read_1, read_2, proper_pair, singleton, mate_mapped,
 * mate_reference_sequence_id_mismatch, .._hq (general/metrics.rs:24-92);
 * out[16..25) read-one CIGAR op counts in BAM op order M I D N S H P = X, out[25..34) read two. */
int ngsq_get_general(ngsq_engine* e, uint64_t out[34]);
int ngsq_get_tlen(ngsq_engine* e, uint64_t hist[1025], uint64_t* processed, uint64_t* ignored);
/* nuc = {gc, at, other}; rec = {processed, ignored_flags, ignored_too_short}.  Window policy for
 * l_seq > 100 (the reference is non-deterministic there, gc_content.rs:69-74):
 * offset = ((splitmix64(gc_seed ^ voffset) >> 32) * (l_seq - 100)) >> 32, voffset = the record's
 * BGZF virtual offset. */
int ngsq_get_gc(ngsq_engine* e, uint64_t hist[101], uint64_t nuc[3], uint64_t rec[3]);
/* out[pos * 94 + score] for pos in [0, *n_positions), *n_positions = longest read with qualities. */
int ngsq_get_quality(ngsq_engine* e, uint64_t* out, size_t cap_positions, uint32_t* n_positions);
typedef struct ngsq_cov_ints {
  uint32_t touched;            /* 1 if pass 2 would have created this contig's entry */
  uint32_t n_bins;             /* entries of mean_coverage_per_bin */
  uint64_t pileup_too_large;   /* positions deeper than 2048 */
  uint64_t hist[2049];         /* depth histogram of positions 0..=L */
} ngsq_cov_ints;
/* bin_sums[k] = sum of depth over the k-th bin of coverage.rs:206-230 (bin 0 = position 0). */
int ngsq_get_coverage_contig(ngsq_engine* e, uint32_t ref, ngsq_cov_ints* out, uint64_t* bin_sums, size_t cap);
int ngsq_get_coverage_global(ngsq_engine* e, uint64_t* nonsensical_records);
/* Edits (edits.rs:22-46): the integer state of EditMetrics when aggregate() runs — read_one_edits / read_two_edits
 * (Histogram 0..=512 of edits per read), vaf_histogram (0..=100, filled by teardown, edits.rs:318-334) and the number
 * of records that were stepped through.  The two means of the summary are the caller's (Histogram::mean). */
/* Genomic Features (features/metrics.rs): utr_five_prime_count, utr_three_prime_count, coding_sequence_count,
 * intergenic_count, exonic_count, intronic_count, processed, ignored_flags, ignored_nonprimary_chromosome. */
int ngsq_get_features(ngsq_engine* e, uint64_t counts[9]);
int ngsq_get_edits(ngsq_engine* e, uint64_t read_one[513], uint64_t read_two[513], uint64_t vaf[101], uint64_t* records);
/* The VAF file of edits.rs:317-340 (`--vaf-file`): refs_per_position / alts_per_position of header sequence `ref` when its
 * teardown runs, n = sequence length + 1 entries each, index = 1-based reference position (alignment_start + reference_ptr,
 * edits.rs:279-281; entry 0 stays 0).  After ngsq_finish; with several engines every engine holds the counts of the records
 * of its own shard (contig-exclusive shards: the owner's are the sequence's; a split reference's counts are the root's once
 * merged, the other engines' are zero). */
int ngsq_get_edit_positions(ngsq_engine* e, uint32_t ref, uint32_t* refs, uint32_t* alts, uint64_t n);
int ngsq_get_stats(ngsq_engine* e, ngsq_stats* out);
/* NGSQ_F_INDEX: the complete .bai file (magic, every reference's bins, chunks, metadata pseudo-bin 37450 and linear index,
 * n_no_coor) of the records submitted since ngsq_set_range.  After ngsq_finish.  *n_out = its size; out = NULL with cap = 0
 * asks for the size only.  DESIGN.md section 4 (K13) lists where its bytes may differ from samtools' index of the same file. */
int ngsq_get_bai(ngsq_engine* e, uint8_t* out, size_t cap, size_t* n_out);
/* NGSQ_F_INDEX_CSI: the binning of the CSI.  min_shift in [12, 24] (windows of 2^min_shift bases); depth in [1, 7], or 0 for
 * the rule of `samtools index -c`: the smallest depth n with (longest reference + 256) <= 2^(min_shift + 3n).  Optional (default
 * 14, 0); before ngsq_set_references, which resolves the depth; kept across ngsq_reset. */
int ngsq_set_index_binning(ngsq_engine* e, uint32_t min_shift, uint32_t depth);
/* NGSQ_F_INDEX | NGSQ_F_INDEX_CSI: the .csi payload, UNCOMPRESSED ("CSI\1", min_shift, depth, l_aux = 0, n_ref; per reference
 * its bins with loffset and chunks and the pseudo-bin n_bins + 1; n_no_coor): the file on disk is this payload BGZF-compressed
 * by the caller.  Conventions of ngsq_get_bai; each of the two refuses an engine of the other format. */
int ngsq_get_csi(ngsq_engine* e, uint8_t* out, size_t cap, size_t* n_out);

/* ---- a BAM without an index cut between engines (DESIGN.md sections 4 K13 and 5) ----
 * Record anchor finder: `bgzf` holds whole BGZF blocks starting at file offset `file_off`.  They are inflated on the device
 * and every offset is tested in parallel for the start of a chain of plausible records (recscan.cuh: plausible()) that runs
 * to the end of the inflated window (its last record may run past it).  *voffset = the smallest such offset as a virtual
 * offset and *ref_id = that record's reference id; *voffset = 0 (and *ref_id = -1) when the window holds none, e.g. when
 * every block lies inside one long read: offer a larger window.  The result is SPECULATIVE: bytes inside a record may look
 * like records.  It is proven only by the closure check of the range that ends there (a range whose end is not a record
 * start fails with NGSQ_E_CHAIN or NGSQ_E_TRUNCATED).  After ngsq_set_references (the test needs n_ref), outside a run. */
int ngsq_find_record(ngsq_engine* e, const uint8_t* bgzf, size_t nbytes, uint64_t file_off, uint64_t* voffset, int32_t* ref_id);
/* Joins the index parts of NGSQ_F_INDEX_PART engines into the file's .bai, on the host (no device work): the same bytes one
 * NGSQ_F_INDEX engine gives for the whole file.  parts[0..n) in file order, each finished without error, all with the same
 * references; part k's end offset equals part k+1's first offset and the last part runs to the end of the data
 * (NGSQ_E_ARG otherwise).  Unsorted records fail with NGSQ_E_UNSORTED and the offset and message one engine gives.  *n_out =
 * the size; out = NULL with cap = 0 asks for the size only.  The message of a failure is ngsq_last_error(parts[0]) (of NULL
 * when parts is NULL or n is 0). */
int ngsq_join_bai(ngsq_engine* const* parts, uint32_t n, uint8_t* out, size_t cap, size_t* n_out);
/* The same for NGSQ_F_INDEX_PART | NGSQ_F_INDEX_CSI parts: the uncompressed .csi one NGSQ_F_INDEX | NGSQ_F_INDEX_CSI engine
 * gives.  Every part must also have the same binning (NGSQ_E_ARG otherwise); BAI parts are refused here, CSI parts by
 * ngsq_join_bai. */
int ngsq_join_csi(ngsq_engine* const* parts, uint32_t n, uint8_t* out, size_t cap, size_t* n_out);

/* ---- multi-GPU merge: one sum-reduce of the packed u64 result buffer ---- */
int ngsq_nccl_unique_id(char out[128]);
int ngsq_comm_init(ngsq_engine* e, int n_ranks, int rank, const char id[128]);
int ngsq_reduce(ngsq_engine* e, int root);
/* Raw access for callers that bring their own collective (bench.py reduces this buffer with
 * torch.distributed): device pointer and length in u64 words.  All ranks must call
 * ngsq_set_quality_positions with the same value (max over ranks) first. */
int ngsq_set_quality_positions(ngsq_engine* e, uint32_t n_positions);
int ngsq_result_buffer(ngsq_engine* e, void** dev_ptr, size_t* n_words);
/* After an external reduction of that buffer: refresh the host copy the ngsq_get_* getters read. */
int ngsq_refresh_results(ngsq_engine* e);

/* ---- shards cut inside a contig (DESIGN.md section 5) ----
 * Reference `ref` is split between shards: this engine scatters into its arrays as usual, but ngsq_finish does not resolve
 * it (K9, and the Edits VAF pass); ngsq_reduce sums every rank's partial arrays of ref onto `root` and resolves it there.
 * Same set on every rank; after ngsq_set_references, before the first submit; kept across ngsq_reset.  Change the set only
 * together with ngsq_set_references on every rank: a rank that adds a reference on its own re-runs the layout agreement of its
 * next ngsq_reduce alone, and the ranks' collectives no longer match.
 * NGSQ_E_ARG with NGSQ_F_INDEX or max_records != 0.  Until the merge, ngsq_get_coverage_contig and ngsq_get_edit_positions
 * of a split reference, and ngsq_get_edits whenever one is declared, fail with NGSQ_E_ARG instead of partial numbers. */
int ngsq_split_reference(ngsq_engine* e, uint32_t ref);

/* Callers that bring their own collective (the pattern of ngsq_result_buffer): the device arrays of a split reference.
 * Valid until the next ngsq_set_references or ngsq_set_quality_positions. */
struct ngsq_split_arrays {
  int32_t*  diff;       uint64_t n_diff;       /* coverage difference array, L + 2 (NULL without NGSQ_F_COVERAGE / mask) */
  int32_t*  tile_sums;  uint64_t n_tiles;      /* its 4096-position tile sums */
  uint64_t* touched;                           /* the contig's touched word */
  uint32_t* edit_refs;  uint32_t* edit_alts;  uint64_t n_positions;  /* L + 1 each (NULL without NGSQ_F_EDITS) */
};
int ngsq_split_arrays(ngsq_engine* e, uint32_t ref, struct ngsq_split_arrays* out);
/* After the caller summed every engine's split arrays element-wise into the root's: the root resolves its split references
 * into its result buffer; every other engine zeroes its split partials (so per-position reads and later sums count once). */
int ngsq_resolve_split(ngsq_engine* e, int is_root);

/* ---- utilities ---- */
void* ngsq_host_alloc(size_t nbytes); /* pinned host memory for ngsq_submit */
void ngsq_host_free(void* p);
/* Page-locks a range the caller already owns (e.g. a mapped file) so that ngsq_submit copies from it asynchronously. */
int ngsq_host_register(void* p, size_t nbytes);
int ngsq_host_unregister(void* p);
/* GPU-inflates whole BGZF blocks and copies the bytes back (header parsing on the host). */
int ngsq_inflate_to_host(ngsq_engine* e, const uint8_t* bgzf, size_t nbytes, uint8_t* out, size_t cap, size_t* n_out);

#ifdef __cplusplus
}
#endif
#endif /* NGS_CUDA_H_ */
