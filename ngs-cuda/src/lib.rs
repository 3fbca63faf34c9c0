//! `ngs-cuda`: the host side of the CUDA engine behind `ngs qc` (include/ngs_cuda.h).
//!
//! NOT COMPILED IN THE ENGINE'S REPOSITORY (its image has no Rust toolchain); every call below is exercised there
//! through the same C ABI by `ngs_b200/host/qc_command.cpp` (C++) and `ngs_b200/ffi.py` (ctypes).
//!
//! What replaces what in `stjude-rust-labs/ngs` v0.4.0:
//!   * `Engine::stream_file` + `Engine::finish`   the two hot loops of `app()`, `src/qc/command.rs:305-316` (pass 1)
//!     and `:350-397` (pass 2), including the BGZF read + inflate + CRC check that `bam::Reader` performs under them
//!     (`src/utils/formats/bam.rs:41-44`);
//!   * `Engine::general()` .. `Engine::coverage_contig()`   the integer state the facets hold when their
//!     `summarize()` / `teardown()` / `aggregate()` run.  Every float stays where it is: in the facets;
//!   * `Engine::create_indexer` + `Engine::build_bai`   the record loop of `ngs index` for a BAM (`src/index/bam.rs:66-100`):
//!     the bytes of the `.bai` from one streamed pass.
//! One `Engine` per GPU, driven by one thread (the qc path is single-threaded: `src/qc.rs:49` uses `Rc`).

use std::ffi::CStr;
use std::fs::File;
use std::io::Read;
use std::os::raw::{c_char, c_int, c_void};
use std::path::Path;

use anyhow::{bail, Context};

pub mod sys {
    //! `extern "C"` declarations, one per entry of include/ngs_cuda.h.
    use super::*;

    #[repr(C)]
    pub struct NgsqEngine {
        _private: [u8; 0],
    }

    #[repr(C)]
    #[derive(Clone, Copy, Default)]
    pub struct NgsqConfig {
        pub struct_size: u32,
        pub flags: u32,
        pub gc_seed: u64,
        pub max_records: u64,
        pub reserve_compressed: u64,
        pub reserve_inflated: u64,
        pub reserve_blocks: u32,
        pub launch_blocks: u32,
        pub quality_positions: u32,
        pub carry_bytes: u32,
        pub comp_ring_bytes: u64,
    }

    #[repr(C)]
    #[derive(Clone, Copy, Default)]
    pub struct NgsqBlock {
        pub coffset: u64,
        pub hdr_len: u32,
        pub csize: u32,
        pub isize: u32,
        pub crc32: u32,
    }

    #[repr(C)]
    #[derive(Clone, Copy, Default)]
    pub struct NgsqStats {
        pub records: u64,
        pub blocks: u64,
        pub compressed_bytes: u64,
        pub inflated_bytes: u64,
        pub max_read_len: u64,
        pub ms_inflate: f32,
        pub ms_crc: f32,
        pub ms_scan: f32,
        pub ms_facets: f32,
        pub ms_coverage: f32,
        pub ms_total: f32,
        pub inflate_launches: u32,
        pub other_launches: u32,
        pub ms_inflate_decode: f32,
        pub ms_inflate_resolve: f32,
        pub ms_reduce: f32,
        pub ms_edits: f32,
        pub ms_tail: f32,
        pub waves: u32,
    }

    #[repr(C)]
    pub struct NgsqCovInts {
        pub touched: u32,
        pub n_bins: u32,
        pub pileup_too_large: u64,
        pub hist: [u64; 2049],
    }

    pub const NGSQ_F_RECORD_FACETS: u32 = 1;
    pub const NGSQ_F_COVERAGE: u32 = 2;
    pub const NGSQ_F_VERIFY_CRC: u32 = 4;
    pub const NGSQ_F_EDITS: u32 = 8;
    pub const NGSQ_F_FEATURES: u32 = 16;
    /// measurement aid: every kernel of a wave on one stream (no overlap with the next wave's inflate); results identical
    pub const NGSQ_F_SERIAL_STAGES: u32 = 32;
    pub const NGSQ_E_QUAL_CAP: c_int = -13;
    pub const NGSQ_F_INDEX: u32 = 64;
    /// index one range of a file cut between engines (set instead of NGSQ_F_INDEX); join the parts with ngsq_join_bai
    pub const NGSQ_F_INDEX_PART: u32 = 128;
    /// with NGSQ_F_INDEX / NGSQ_F_INDEX_PART: a CSI instead of a BAI (ngsq_get_csi, ngsq_join_csi)
    pub const NGSQ_F_INDEX_CSI: u32 = 256;
    pub const NGSQ_E_UNSORTED: c_int = -14;

    /// Device arrays of a reference split between shards (`struct ngsq_split_arrays`); null pointers for facets that are off.
    #[repr(C)]
    #[derive(Clone, Copy, Debug)]
    pub struct NgsqSplitArrays {
        pub diff: *mut i32,
        pub n_diff: u64,
        pub tile_sums: *mut i32,
        pub n_tiles: u64,
        pub touched: *mut u64,
        pub edit_refs: *mut u32,
        pub edit_alts: *mut u32,
        pub n_positions: u64,
    }

    extern "C" {
        pub fn ngsq_version() -> c_int;
        pub fn ngsq_last_error(e: *mut NgsqEngine) -> *const c_char;
        pub fn ngsq_create(device: c_int, cfg: *const NgsqConfig, out: *mut *mut NgsqEngine) -> c_int;
        pub fn ngsq_destroy(e: *mut NgsqEngine);
        pub fn ngsq_reset(e: *mut NgsqEngine) -> c_int;
        pub fn ngsq_set_references(e: *mut NgsqEngine, n_ref: u32, ref_len: *const u32, coverage_enabled: *const u8) -> c_int;
        pub fn ngsq_set_reference_bases(e: *mut NgsqEngine, r: u32, letters: *const u8, n: u64) -> c_int;
        pub fn ngsq_set_feature_model(e: *mut NgsqEngine, slot_class: *const u8, primary: *const u8) -> c_int;
        pub fn ngsq_set_features(e: *mut NgsqEngine, r: u32, n: u32, start: *const u32, stop: *const u32, cls: *const u8) -> c_int;
        pub fn ngsq_set_range(e: *mut NgsqEngine, first_rec_voffset: u64, end_voffset: u64) -> c_int;
        pub fn ngsq_bgzf_walk(bgzf: *const u8, nbytes: usize, file_off: u64, out: *mut NgsqBlock, cap: u32, n_blocks: *mut u32, consumed: *mut usize) -> c_int;
        pub fn ngsq_submit(e: *mut NgsqEngine, bgzf: *const u8, nbytes: usize, file_off: u64) -> c_int;
        pub fn ngsq_flush(e: *mut NgsqEngine) -> c_int;
        pub fn ngsq_progress(e: *mut NgsqEngine, records: *mut u64) -> c_int;
        pub fn ngsq_wait_copied(e: *mut NgsqEngine, submit_index: u32) -> c_int;
        pub fn ngsq_submit_device(e: *mut NgsqEngine, dev_bgzf: *const c_void, nbytes: usize, blocks: *const NgsqBlock, n_blocks: u32) -> c_int;
        pub fn ngsq_finish(e: *mut NgsqEngine) -> c_int;
        pub fn ngsq_get_general(e: *mut NgsqEngine, out: *mut u64) -> c_int;
        pub fn ngsq_get_tlen(e: *mut NgsqEngine, hist: *mut u64, processed: *mut u64, ignored: *mut u64) -> c_int;
        pub fn ngsq_get_gc(e: *mut NgsqEngine, hist: *mut u64, nuc: *mut u64, rec: *mut u64) -> c_int;
        pub fn ngsq_get_quality(e: *mut NgsqEngine, out: *mut u64, cap_positions: usize, n_positions: *mut u32) -> c_int;
        pub fn ngsq_get_coverage_contig(e: *mut NgsqEngine, r: u32, out: *mut NgsqCovInts, bin_sums: *mut u64, cap: usize) -> c_int;
        pub fn ngsq_get_coverage_global(e: *mut NgsqEngine, nonsensical_records: *mut u64) -> c_int;
        pub fn ngsq_get_features(e: *mut NgsqEngine, counts: *mut u64) -> c_int;
        pub fn ngsq_get_edits(e: *mut NgsqEngine, read_one: *mut u64, read_two: *mut u64, vaf: *mut u64, records: *mut u64) -> c_int;
        pub fn ngsq_get_edit_positions(e: *mut NgsqEngine, r: u32, refs: *mut u32, alts: *mut u32, n: u64) -> c_int;
        pub fn ngsq_get_stats(e: *mut NgsqEngine, out: *mut NgsqStats) -> c_int;
        pub fn ngsq_nccl_unique_id(out: *mut c_char) -> c_int;
        pub fn ngsq_comm_init(e: *mut NgsqEngine, n_ranks: c_int, rank: c_int, id: *const c_char) -> c_int;
        pub fn ngsq_reduce(e: *mut NgsqEngine, root: c_int) -> c_int;
        pub fn ngsq_set_quality_positions(e: *mut NgsqEngine, n_positions: u32) -> c_int;
        pub fn ngsq_result_buffer(e: *mut NgsqEngine, dev_ptr: *mut *mut c_void, n_words: *mut usize) -> c_int;
        pub fn ngsq_refresh_results(e: *mut NgsqEngine) -> c_int;
        pub fn ngsq_host_alloc(nbytes: usize) -> *mut c_void;
        pub fn ngsq_host_free(p: *mut c_void);
        pub fn ngsq_host_register(p: *mut c_void, nbytes: usize) -> c_int;
        pub fn ngsq_host_unregister(p: *mut c_void) -> c_int;
        pub fn ngsq_get_bai(e: *mut NgsqEngine, out: *mut u8, cap: usize, n_out: *mut usize) -> c_int;
        pub fn ngsq_inflate_to_host(e: *mut NgsqEngine, bgzf: *const u8, nbytes: usize, out: *mut u8, cap: usize, n_out: *mut usize) -> c_int;
        pub fn ngsq_split_reference(e: *mut NgsqEngine, r: u32) -> c_int;
        pub fn ngsq_split_arrays(e: *mut NgsqEngine, r: u32, out: *mut NgsqSplitArrays) -> c_int;
        pub fn ngsq_resolve_split(e: *mut NgsqEngine, is_root: c_int) -> c_int;
        pub fn ngsq_find_record(e: *mut NgsqEngine, bgzf: *const u8, nbytes: usize, file_off: u64, voffset: *mut u64, ref_id: *mut i32) -> c_int;
        pub fn ngsq_join_bai(parts: *const *mut NgsqEngine, n: u32, out: *mut u8, cap: usize, n_out: *mut usize) -> c_int;
        pub fn ngsq_set_index_binning(e: *mut NgsqEngine, min_shift: u32, depth: u32) -> c_int;
        pub fn ngsq_get_csi(e: *mut NgsqEngine, out: *mut u8, cap: usize, n_out: *mut usize) -> c_int;
        pub fn ngsq_join_csi(parts: *const *mut NgsqEngine, n: u32, out: *mut u8, cap: usize, n_out: *mut usize) -> c_int;
    }
}

/// Which facets the engine computes (`get_qc_facets`, `src/qc.rs:49-134`, decides; this is its answer as a bit mask).
#[derive(Clone, Copy, Debug, Default)]
pub struct Facets {
    /// General, Template Length, GC Content, Quality Score.
    pub record_defaults: bool,
    pub coverage: bool,
    pub edits: bool,
    pub features: bool,
}

/// Integer state of `CoverageFacet` for one reference sequence after the second pass.
pub struct CoverageContig {
    /// `coverage_per_position` holds an entry for this sequence (`coverage.rs:155-163`).
    pub touched: bool,
    pub pileup_too_large_positions: u64,
    /// Depth histogram of positions `0..=L`, bins `0..=2048` (`coverage.rs:198-212`).
    pub coverages: Vec<u64>,
    /// Sum of depth over every bin of `coverage.rs:206-230`; the caller divides (f64) by the bin size / the tail modulo.
    pub bin_sums: Vec<u64>,
}

/// Pinned host buffer (cudaHostAlloc): the source of an asynchronous host-to-device copy.
struct Pinned {
    ptr: *mut u8,
    len: usize,
}
impl Pinned {
    fn new(len: usize) -> anyhow::Result<Self> {
        let ptr = unsafe { sys::ngsq_host_alloc(len) } as *mut u8;
        if ptr.is_null() {
            bail!("ngs-cuda: cannot allocate {} bytes of pinned host memory", len);
        }
        Ok(Self { ptr, len })
    }
    fn as_mut(&mut self) -> &mut [u8] {
        unsafe { std::slice::from_raw_parts_mut(self.ptr, self.len) }
    }
}
impl Drop for Pinned {
    fn drop(&mut self) {
        unsafe { sys::ngsq_host_free(self.ptr as *mut c_void) }
    }
}

pub struct Engine {
    raw: *mut sys::NgsqEngine,
    submits: u32,
}

impl Engine {
    /// `num_records`: `-n` (`NumberOfRecords::Some`), 0 = all.  `gc_seed`: the GC window policy (include/ngs_cuda.h,
    /// `ngsq_get_gc`): the reference draws the window offset from an OS-seeded RNG (`gc_content.rs:69-74`).
    pub fn create(device: i32, facets: Facets, num_records: u64, gc_seed: u64) -> anyhow::Result<Self> {
        let mut flags = sys::NGSQ_F_VERIFY_CRC; // noodles-bgzf checks every block's CRC32
        if facets.record_defaults { flags |= sys::NGSQ_F_RECORD_FACETS; }
        if facets.coverage { flags |= sys::NGSQ_F_COVERAGE; }
        if facets.edits { flags |= sys::NGSQ_F_EDITS; }
        if facets.features { flags |= sys::NGSQ_F_FEATURES; }
        let cfg = sys::NgsqConfig { struct_size: std::mem::size_of::<sys::NgsqConfig>() as u32, flags, gc_seed, max_records: num_records, ..Default::default() };
        let mut raw = std::ptr::null_mut();
        let rc = unsafe { sys::ngsq_create(device as c_int, &cfg, &mut raw) };
        if rc != 0 {
            let msg = unsafe { CStr::from_ptr(sys::ngsq_last_error(std::ptr::null_mut())) }.to_string_lossy().into_owned();
            bail!("ngs-cuda: {}", msg); // no CUDA device: there is no CPU fallback, the caller keeps its CPU path
        }
        Ok(Self { raw, submits: 0 })
    }

    fn check(&self, rc: c_int) -> anyhow::Result<()> {
        if rc == 0 {
            return Ok(());
        }
        let msg = unsafe { CStr::from_ptr(sys::ngsq_last_error(self.raw)) }.to_string_lossy().into_owned();
        bail!("ngs-cuda: {}", msg) // NGSQ_E_* map onto the anyhow errors app() already returns
    }

    /// Lengths of the header's reference sequences, in header order, and `supports_sequence_name` of the Coverage facet.
    pub fn set_references(&mut self, lengths: &[u32], coverage_enabled: &[bool]) -> anyhow::Result<()> {
        assert_eq!(lengths.len(), coverage_enabled.len());
        let en: Vec<u8> = coverage_enabled.iter().map(|&b| b as u8).collect();
        self.check(unsafe { sys::ngsq_set_references(self.raw, lengths.len() as u32, lengths.as_ptr(), en.as_ptr()) })
    }

    /// Virtual offsets of the first record this engine owns (`reader.virtual_position()` after the header for a whole
    /// file) and of the first record it does not own (0 = to the end).
    pub fn set_range(&mut self, first: u64, end: u64) -> anyhow::Result<()> {
        self.check(unsafe { sys::ngsq_set_range(self.raw, first, end) })
    }

    /// Streams file bytes `[lo, hi)` (`lo` on a BGZF block boundary) through a ring of three pinned buffers: the read
    /// of chunk k+2, the PCIe copy of chunk k+1 and the kernels of chunk k overlap.  `on_progress(records)` is called
    /// after every chunk with the number of records scanned so far (`RecordCounter`, `src/utils/display.rs:43-52`).
    pub fn stream_file(&mut self, path: &Path, lo: u64, hi: u64, chunk_bytes: usize, mut on_progress: impl FnMut(u64)) -> anyhow::Result<()> {
        use std::io::{Seek, SeekFrom};
        const LEAD: usize = 1 << 17; // room for the previous chunk's partial block
        let mut file = File::open(path).with_context(|| format!("opening {}", path.display()))?;
        file.seek(SeekFrom::Start(lo))?;
        let mut bufs = [Pinned::new(LEAD + chunk_bytes)?, Pinned::new(LEAD + chunk_bytes)?, Pinned::new(LEAD + chunk_bytes)?];
        let mut used_by: [Option<u32>; 3] = [None; 3];
        let mut carry: Vec<u8> = Vec::new();
        let (mut pos, mut file_off, mut k) = (lo, lo, 0usize);
        while pos < hi {
            let bi = k % 3;
            if let Some(idx) = used_by[bi] {
                self.check(unsafe { sys::ngsq_wait_copied(self.raw, idx) })?; // its last copy must have left the buffer
            }
            let want = chunk_bytes.min((hi - pos) as usize);
            let buf = bufs[bi].as_mut();
            let begin = LEAD - carry.len();
            buf[begin..LEAD].copy_from_slice(&carry);
            let mut got = 0;
            while got < want {
                let n = file.read(&mut buf[LEAD + got..LEAD + want])?;
                if n == 0 { break; }
                got += n;
            }
            pos += got as u64;
            let n = carry.len() + got;
            let last = pos >= hi || got < want;
            let (mut nb, mut used) = (0u32, 0usize);
            let rc = unsafe { sys::ngsq_bgzf_walk(buf[begin..].as_ptr(), n, file_off, std::ptr::null_mut(), 0, &mut nb, &mut used) };
            if rc != 0 { bail!("malformed BGZF framing at file offset {}", file_off); }
            if last && used != n { bail!("truncated BGZF block at end of file"); }
            if used > 0 {
                self.check(unsafe { sys::ngsq_submit(self.raw, buf[begin..].as_ptr(), used, file_off) })?;
                used_by[bi] = Some(self.submits);
                self.submits += 1;
                file_off += used as u64;
            }
            carry = buf[begin + used..begin + n].to_vec();
            if carry.len() > LEAD { bail!("BGZF block larger than 128 KiB"); }
            let mut records = 0u64;
            self.check(unsafe { sys::ngsq_progress(self.raw, &mut records) })?;
            on_progress(records);
            if got < want { break; }
            k += 1;
        }
        Ok(())
    }

    /// Last wave, coverage resolve, result read-back.  Replaces the loops at `command.rs:305-316` and `:350-397`.
    pub fn finish(&mut self) -> anyhow::Result<sys::NgsqStats> {
        self.check(unsafe { sys::ngsq_finish(self.raw) })?;
        let mut st = sys::NgsqStats::default();
        self.check(unsafe { sys::ngsq_get_stats(self.raw, &mut st) })?;
        Ok(st)
    }

    /// An engine that builds the BAI of a whole coordinate-sorted BAM (NGSQ_F_INDEX, CRC checked like noodles-bgzf does).
    pub fn create_indexer(device: i32) -> anyhow::Result<Self> {
        let cfg = sys::NgsqConfig {
            struct_size: std::mem::size_of::<sys::NgsqConfig>() as u32,
            flags: sys::NGSQ_F_INDEX | sys::NGSQ_F_VERIFY_CRC,
            ..Default::default()
        };
        let mut raw = std::ptr::null_mut();
        let rc = unsafe { sys::ngsq_create(device as c_int, &cfg, &mut raw) };
        if rc != 0 {
            let msg = unsafe { CStr::from_ptr(sys::ngsq_last_error(std::ptr::null_mut())) }.to_string_lossy().into_owned();
            bail!("ngs-cuda: {}", msg);
        }
        Ok(Self { raw, submits: 0 })
    }

    /// The `.bai` bytes of the BAM at `path` (`src/index/bam.rs:66-100`): `lengths` are the header's reference lengths and
    /// `first_record` the reader's virtual position after the header.  Unsorted records fail (NGSQ_E_UNSORTED), like the
    /// reference's indexer; references of 2^29 bases or more need CSI and are refused.
    pub fn build_bai(&mut self, path: &Path, lengths: &[u32], first_record: u64, chunk_bytes: usize, on_progress: impl FnMut(u64)) -> anyhow::Result<Vec<u8>> {
        self.set_references(lengths, &vec![false; lengths.len()])?;
        self.set_range(first_record, 0)?;
        let size = std::fs::metadata(path)?.len();
        self.stream_file(path, first_record >> 16, size, chunk_bytes, on_progress)?;
        self.finish()?;
        let mut n = 0usize;
        self.check(unsafe { sys::ngsq_get_bai(self.raw, std::ptr::null_mut(), 0, &mut n) })?;
        let mut out = vec![0u8; n];
        self.check(unsafe { sys::ngsq_get_bai(self.raw, out.as_mut_ptr(), out.len(), &mut n) })?;
        Ok(out)
    }

    /// An engine that builds the CSI of a whole coordinate-sorted BAM (NGSQ_F_INDEX | NGSQ_F_INDEX_CSI) at `min_shift`, the
    /// depth by samtools' rule.
    pub fn create_csi_indexer(device: i32, min_shift: u32) -> anyhow::Result<Self> {
        let cfg = sys::NgsqConfig {
            struct_size: std::mem::size_of::<sys::NgsqConfig>() as u32,
            flags: sys::NGSQ_F_INDEX | sys::NGSQ_F_INDEX_CSI | sys::NGSQ_F_VERIFY_CRC,
            ..Default::default()
        };
        let mut raw = std::ptr::null_mut();
        let rc = unsafe { sys::ngsq_create(device as c_int, &cfg, &mut raw) };
        if rc != 0 {
            let msg = unsafe { CStr::from_ptr(sys::ngsq_last_error(std::ptr::null_mut())) }.to_string_lossy().into_owned();
            bail!("ngs-cuda: {}", msg);
        }
        let mut e = Self { raw, submits: 0 };
        e.check(unsafe { sys::ngsq_set_index_binning(e.raw, min_shift, 0) })?;
        Ok(e)
    }

    /// The UNCOMPRESSED `.csi` payload of the BAM at `path` (an engine of `create_csi_indexer`); the file on disk is its BGZF
    /// compression.  Arguments and refusals as `build_bai`, with the CSI's limit 2^(min_shift + 3 depth).
    pub fn build_csi(&mut self, path: &Path, lengths: &[u32], first_record: u64, chunk_bytes: usize, on_progress: impl FnMut(u64)) -> anyhow::Result<Vec<u8>> {
        self.set_references(lengths, &vec![false; lengths.len()])?;
        self.set_range(first_record, 0)?;
        let size = std::fs::metadata(path)?.len();
        self.stream_file(path, first_record >> 16, size, chunk_bytes, on_progress)?;
        self.finish()?;
        let mut n = 0usize;
        self.check(unsafe { sys::ngsq_get_csi(self.raw, std::ptr::null_mut(), 0, &mut n) })?;
        let mut out = vec![0u8; n];
        self.check(unsafe { sys::ngsq_get_csi(self.raw, out.as_mut_ptr(), out.len(), &mut n) })?;
        Ok(out)
    }

    /// An engine that indexes one range of a file cut between engines (NGSQ_F_INDEX_PART beside `flags`, e.g. the qc flags);
    /// its part is joined with the others by `join_bai` after `finish`.
    pub fn create_index_part(device: i32, flags: u32) -> anyhow::Result<Self> {
        let cfg = sys::NgsqConfig {
            struct_size: std::mem::size_of::<sys::NgsqConfig>() as u32,
            flags: flags | sys::NGSQ_F_INDEX_PART,
            ..Default::default()
        };
        let mut raw = std::ptr::null_mut();
        let rc = unsafe { sys::ngsq_create(device as c_int, &cfg, &mut raw) };
        if rc != 0 {
            let msg = unsafe { CStr::from_ptr(sys::ngsq_last_error(std::ptr::null_mut())) }.to_string_lossy().into_owned();
            bail!("ngs-cuda: {}", msg);
        }
        Ok(Self { raw, submits: 0 })
    }

    /// The first record start in whole BGZF blocks `bgzf` that begin at file offset `file_off`, as (virtual offset, reference
    /// id); None when the window holds none (offer a larger one).  Speculative: the range that ends there proves it.
    pub fn find_record(&mut self, bgzf: &[u8], file_off: u64) -> anyhow::Result<Option<(u64, i32)>> {
        let (mut v, mut r) = (0u64, -1i32);
        self.check(unsafe { sys::ngsq_find_record(self.raw, bgzf.as_ptr(), bgzf.len(), file_off, &mut v, &mut r) })?;
        Ok(if v == 0 { None } else { Some((v, r)) })
    }

    /// A read longer than the quality table: raise it and run the file again (include/ngs_cuda.h, NGSQ_E_QUAL_CAP).
    pub fn set_quality_positions(&mut self, n: u32) -> anyhow::Result<()> {
        self.check(unsafe { sys::ngsq_set_quality_positions(self.raw, n) })
    }
    pub fn reset(&mut self) -> anyhow::Result<()> {
        self.submits = 0;
        self.check(unsafe { sys::ngsq_reset(self.raw) })
    }

    // ---- integer getters (valid after finish / reduce) ----
    /// `[0..16)` RecordMetrics in declaration order (`general/metrics.rs:24-92`), `[16..25)` read-one CIGAR op counts in
    /// BAM op order `M I D N S H P = X`, `[25..34)` read two.
    pub fn general(&self) -> anyhow::Result<[u64; 34]> {
        let mut g = [0u64; 34];
        self.check(unsafe { sys::ngsq_get_general(self.raw, g.as_mut_ptr()) })?;
        Ok(g)
    }
    /// (histogram `0..=1024`, processed, ignored) of `TemplateLengthFacet` (`template_length.rs:43-53`).
    pub fn template_length(&self) -> anyhow::Result<(Vec<u64>, u64, u64)> {
        let mut h = vec![0u64; 1025];
        let (mut p, mut i) = (0u64, 0u64);
        self.check(unsafe { sys::ngsq_get_tlen(self.raw, h.as_mut_ptr(), &mut p, &mut i) })?;
        Ok((h, p, i))
    }
    /// (histogram `0..=100`, `[gc, at, other]`, `[processed, ignored_flags, ignored_too_short]`) of `GCContentMetrics`.
    pub fn gc_content(&self) -> anyhow::Result<(Vec<u64>, [u64; 3], [u64; 3])> {
        let mut h = vec![0u64; 101];
        let (mut nuc, mut rec) = ([0u64; 3], [0u64; 3]);
        self.check(unsafe { sys::ngsq_get_gc(self.raw, h.as_mut_ptr(), nuc.as_mut_ptr(), rec.as_mut_ptr()) })?;
        Ok((h, nuc, rec))
    }
    /// `scores[pos][q]` for `pos < n_positions`: `QualityScoreFacet::scores` holds key `pos + 1` (`quality_scores.rs:37-49`).
    pub fn quality_scores(&self) -> anyhow::Result<Vec<[u64; 94]>> {
        let mut n = 0u32;
        self.check(unsafe { sys::ngsq_get_quality(self.raw, std::ptr::null_mut(), 0, &mut n) })?;
        let mut out = vec![[0u64; 94]; n as usize];
        if n > 0 {
            self.check(unsafe { sys::ngsq_get_quality(self.raw, out.as_mut_ptr() as *mut u64, n as usize, &mut n) })?;
        }
        Ok(out)
    }
    pub fn coverage_contig(&self, reference: u32, length: u32) -> anyhow::Result<CoverageContig> {
        let mut ints = Box::new(sys::NgsqCovInts { touched: 0, n_bins: 0, pileup_too_large: 0, hist: [0; 2049] });
        let cap = length as usize / 50_000 + 3;
        let mut bins = vec![0u64; cap];
        self.check(unsafe { sys::ngsq_get_coverage_contig(self.raw, reference, &mut *ints, bins.as_mut_ptr(), cap) })?;
        bins.truncate(ints.n_bins as usize);
        Ok(CoverageContig { touched: ints.touched != 0, pileup_too_large_positions: ints.pileup_too_large, coverages: ints.hist.to_vec(), bin_sums: bins })
    }
    pub fn nonsensical_records(&self) -> anyhow::Result<u64> {
        let mut v = 0u64;
        self.check(unsafe { sys::ngsq_get_coverage_global(self.raw, &mut v) })?;
        Ok(v)
    }

    // ---- Edits / Genomic Features (Facets { edits, features }) ----
    /// `EditsFacet::setup` for header sequence `reference`: the letters of its FASTA record (`edits.rs:186-207`).  After
    /// `set_references`, before the first chunk.
    pub fn set_reference_bases(&mut self, reference: u32, letters: &[u8]) -> anyhow::Result<()> {
        self.check(unsafe { sys::ngsq_set_reference_bases(self.raw, reference, letters.as_ptr(), letters.len() as u64) })
    }
    /// `slot_class[j]` = first of the five configured feature names (5' UTR, 3' UTR, CDS, exon, gene) equal to name j;
    /// `primary[c]` = header sequence c belongs to the genome's primary assembly (`features.rs:131-140`, `:287-345`).
    pub fn set_feature_model(&mut self, slot_class: &[u8], primary: &[u8]) -> anyhow::Result<()> {
        if slot_class.len() != 5 {
            bail!("ngs-cuda: five feature names expected");
        }
        self.check(unsafe { sys::ngsq_set_feature_model(self.raw, slot_class.as_ptr(), primary.as_ptr()) })
    }
    /// The kept GFF records of one header sequence: start, end as in the GFF, slot of their type.
    pub fn set_features(&mut self, reference: u32, start: &[u32], stop: &[u32], class: &[u8]) -> anyhow::Result<()> {
        if start.len() != stop.len() || start.len() != class.len() {
            bail!("ngs-cuda: feature arrays differ in length");
        }
        self.check(unsafe { sys::ngsq_set_features(self.raw, reference, start.len() as u32, start.as_ptr(), stop.as_ptr(), class.as_ptr()) })
    }
    /// (read_one_edits `0..=512`, read_two_edits `0..=512`, vaf_histogram `0..=100`, records stepped through) of `EditMetrics`
    /// when `aggregate()` runs (`edits.rs:22-46`, `:336-344`).
    pub fn edits(&self) -> anyhow::Result<(Vec<u64>, Vec<u64>, Vec<u64>, u64)> {
        let (mut one, mut two, mut vaf, mut n) = (vec![0u64; 513], vec![0u64; 513], vec![0u64; 101], 0u64);
        self.check(unsafe { sys::ngsq_get_edits(self.raw, one.as_mut_ptr(), two.as_mut_ptr(), vaf.as_mut_ptr(), &mut n) })?;
        Ok((one, two, vaf, n))
    }
    /// `refs_per_position` / `alts_per_position` of one header sequence at its teardown, indexed by 1-based position: what
    /// `EditsFacet::teardown` iterates to write the VAF file (`edits.rs:317-340`).
    pub fn edit_positions(&self, reference: u32, length: u32) -> anyhow::Result<(Vec<u32>, Vec<u32>)> {
        let n = length as usize + 1;
        let (mut refs, mut alts) = (vec![0u32; n], vec![0u32; n]);
        self.check(unsafe { sys::ngsq_get_edit_positions(self.raw, reference, refs.as_mut_ptr(), alts.as_mut_ptr(), n as u64) })?;
        Ok((refs, alts))
    }
    /// The nine counters of `GenomicFeaturesMetrics` in declaration order (`features/metrics.rs`).
    pub fn features(&self) -> anyhow::Result<[u64; 9]> {
        let mut c = [0u64; 9];
        self.check(unsafe { sys::ngsq_get_features(self.raw, c.as_mut_ptr()) })?;
        Ok(c)
    }

    // ---- multi-GPU: one Engine per device and thread, shards cut at the BAI's per-reference extents ----
    pub fn nccl_unique_id() -> anyhow::Result<[c_char; 128]> {
        let mut id = [0 as c_char; 128];
        if unsafe { sys::ngsq_nccl_unique_id(id.as_mut_ptr()) } != 0 {
            bail!("ngs-cuda: ncclGetUniqueId failed");
        }
        Ok(id)
    }
    pub fn comm_init(&mut self, n_ranks: i32, rank: i32, id: &[c_char; 128]) -> anyhow::Result<()> {
        self.check(unsafe { sys::ngsq_comm_init(self.raw, n_ranks, rank, id.as_ptr()) })
    }
    /// ONE sum all-reduce of the packed integer results (after every engine's `finish`); references declared with
    /// `split_reference` are summed onto `root` and resolved there first.
    pub fn reduce(&mut self, root: i32) -> anyhow::Result<()> {
        self.check(unsafe { sys::ngsq_reduce(self.raw, root) })
    }

    // ---- shards cut inside a contig (DESIGN.md section 5) ----
    /// Declares reference `r` split between shards: the same set on every engine, after `set_references`, before the first
    /// submit.  Its coverage and VAF counters are resolved by `reduce` (or `resolve_split`), not by `finish`.  With records in
    /// any order (`--cuda-any-order` on several devices) every reference of the header is declared: any contig can have
    /// records on both sides of any cut.
    pub fn split_reference(&mut self, r: u32) -> anyhow::Result<()> {
        self.check(unsafe { sys::ngsq_split_reference(self.raw, r) })
    }
    /// The device arrays of a split reference, for a caller that sums them with its own collective.
    pub fn split_arrays(&mut self, r: u32) -> anyhow::Result<sys::NgsqSplitArrays> {
        let mut out = sys::NgsqSplitArrays {
            diff: std::ptr::null_mut(),
            n_diff: 0,
            tile_sums: std::ptr::null_mut(),
            n_tiles: 0,
            touched: std::ptr::null_mut(),
            edit_refs: std::ptr::null_mut(),
            edit_alts: std::ptr::null_mut(),
            n_positions: 0,
        };
        self.check(unsafe { sys::ngsq_split_arrays(self.raw, r, &mut out) })?;
        Ok(out)
    }
    /// After the split arrays of every engine were summed into the root's: resolve them on the root, zero them elsewhere.
    pub fn resolve_split(&mut self, is_root: bool) -> anyhow::Result<()> {
        self.check(unsafe { sys::ngsq_resolve_split(self.raw, is_root as c_int) })
    }
}

/// The `.bai` of a file from its finished NGSQ_F_INDEX_PART engines, in file order (ngsq_join_bai, on the host).
pub fn join_bai(parts: &[&Engine]) -> anyhow::Result<Vec<u8>> {
    if parts.is_empty() {
        bail!("ngs-cuda: join_bai needs at least one part");
    }
    let raws: Vec<*mut sys::NgsqEngine> = parts.iter().map(|e| e.raw).collect();
    let mut n = 0usize;
    parts[0].check(unsafe { sys::ngsq_join_bai(raws.as_ptr(), raws.len() as u32, std::ptr::null_mut(), 0, &mut n) })?;
    let mut out = vec![0u8; n];
    parts[0].check(unsafe { sys::ngsq_join_bai(raws.as_ptr(), raws.len() as u32, out.as_mut_ptr(), out.len(), &mut n) })?;
    Ok(out)
}

/// The uncompressed `.csi` of a file from its finished NGSQ_F_INDEX_PART | NGSQ_F_INDEX_CSI engines, in file order
/// (ngsq_join_csi; every part must have the same binning).
pub fn join_csi(parts: &[&Engine]) -> anyhow::Result<Vec<u8>> {
    if parts.is_empty() {
        bail!("ngs-cuda: join_csi needs at least one part");
    }
    let raws: Vec<*mut sys::NgsqEngine> = parts.iter().map(|e| e.raw).collect();
    let mut n = 0usize;
    parts[0].check(unsafe { sys::ngsq_join_csi(raws.as_ptr(), raws.len() as u32, std::ptr::null_mut(), 0, &mut n) })?;
    let mut out = vec![0u8; n];
    parts[0].check(unsafe { sys::ngsq_join_csi(raws.as_ptr(), raws.len() as u32, out.as_mut_ptr(), out.len(), &mut n) })?;
    Ok(out)
}

impl Drop for Engine {
    fn drop(&mut self) {
        unsafe { sys::ngsq_destroy(self.raw) }
    }
}

// One engine is driven by one thread, but it may be created on one and moved to another (one thread per GPU).
unsafe impl Send for Engine {}
