"""ctypes binding of libngs_cuda.so — the same symbols a Rust `ngs-cuda` module would bind
(include/ngs_cuda.h; INTEGRATION.md shows the `extern "C"` block).

There is no CPU path: if the CUDA library is missing or no device is present this module
raises instead of falling back.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libngs_cuda.so")
SYNTH_PATH = os.path.join(_HERE, "libngs_synth.so")

NGSQ_F_RECORD_FACETS = 1
NGSQ_F_COVERAGE = 2
NGSQ_F_VERIFY_CRC = 4
NGSQ_F_EDITS = 8
NGSQ_F_FEATURES = 16
NGSQ_F_SERIAL_STAGES = 32  # measurement aid: no overlap between the stages of consecutive waves
NGSQ_F_INDEX = 64  # build the file's BAI in the same pass (Engine.bai())
NGSQ_F_INDEX_PART = 128  # index one range of a file cut between engines (join the parts with join_bai())
NGSQ_F_INDEX_CSI = 256  # with NGSQ_F_INDEX / NGSQ_F_INDEX_PART: a CSI instead of a BAI (Engine.csi(), join_csi())

ERROR_NAMES = {
    0: "NGSQ_OK", -1: "NGSQ_E_ARG", -2: "NGSQ_E_CUDA", -3: "NGSQ_E_TRUNCATED", -4: "NGSQ_E_BAD_BLOCK",
    -5: "NGSQ_E_CRC", -6: "NGSQ_E_BAD_RECORD", -7: "NGSQ_E_QUAL_RANGE", -8: "NGSQ_E_CHAIN",
    -9: "NGSQ_E_NCCL", -10: "NGSQ_E_NOMEM", -11: "NGSQ_E_EDITS", -12: "NGSQ_E_FEATURES", -13: "NGSQ_E_QUAL_CAP",
    -14: "NGSQ_E_UNSORTED",
}

# every symbol include/ngs_cuda.h declares (tests check the library exports all of them)
EXPORTED = [
    "ngsq_version", "ngsq_last_error", "ngsq_create", "ngsq_destroy", "ngsq_reset", "ngsq_set_references",
    "ngsq_set_range", "ngsq_bgzf_walk", "ngsq_submit", "ngsq_submit_device", "ngsq_finish", "ngsq_get_general",
    "ngsq_get_tlen", "ngsq_get_gc", "ngsq_get_quality", "ngsq_get_coverage_contig", "ngsq_get_coverage_global",
    "ngsq_get_stats", "ngsq_nccl_unique_id", "ngsq_comm_init", "ngsq_reduce", "ngsq_set_quality_positions",
    "ngsq_result_buffer", "ngsq_refresh_results", "ngsq_host_alloc", "ngsq_host_free", "ngsq_inflate_to_host",
    "ngsq_set_reference_bases", "ngsq_get_edits", "ngsq_get_edit_positions", "ngsq_set_feature_model", "ngsq_set_features", "ngsq_get_features",
    "ngsq_wait_copied", "ngsq_host_register", "ngsq_host_unregister", "ngsq_flush", "ngsq_progress",
    "ngsq_get_bai", "ngsq_split_reference", "ngsq_split_arrays", "ngsq_resolve_split", "ngsq_find_record", "ngsq_join_bai",
    "ngsq_set_index_binning", "ngsq_get_csi", "ngsq_join_csi",
]


class NgsqError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"{ERROR_NAMES.get(code, code)}: {message}")
        self.code = code


class Config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("flags", C.c_uint32), ("gc_seed", C.c_uint64), ("max_records", C.c_uint64),
        ("reserve_compressed", C.c_uint64), ("reserve_inflated", C.c_uint64), ("reserve_blocks", C.c_uint32),
        ("launch_blocks", C.c_uint32), ("quality_positions", C.c_uint32), ("carry_bytes", C.c_uint32), ("comp_ring_bytes", C.c_uint64),
    ]


class Block(C.Structure):
    _fields_ = [("coffset", C.c_uint64), ("hdr_len", C.c_uint32), ("csize", C.c_uint32), ("isize", C.c_uint32),
                ("crc32", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [
        ("records", C.c_uint64), ("blocks", C.c_uint64), ("compressed_bytes", C.c_uint64), ("inflated_bytes", C.c_uint64),
        ("max_read_len", C.c_uint64), ("ms_inflate", C.c_float), ("ms_crc", C.c_float), ("ms_scan", C.c_float),
        ("ms_facets", C.c_float), ("ms_coverage", C.c_float), ("ms_total", C.c_float), ("inflate_launches", C.c_uint32),
        ("other_launches", C.c_uint32), ("ms_inflate_decode", C.c_float), ("ms_inflate_resolve", C.c_float), ("ms_reduce", C.c_float),
        ("ms_edits", C.c_float), ("ms_tail", C.c_float), ("waves", C.c_uint32),
    ]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class SplitArrays(C.Structure):
    _fields_ = [("diff", C.c_void_p), ("n_diff", C.c_uint64), ("tile_sums", C.c_void_p), ("n_tiles", C.c_uint64),
                ("touched", C.c_void_p), ("edit_refs", C.c_void_p), ("edit_alts", C.c_void_p), ("n_positions", C.c_uint64)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class CovInts(C.Structure):
    _fields_ = [("touched", C.c_uint32), ("n_bins", C.c_uint32), ("pileup_too_large", C.c_uint64), ("hist", C.c_uint64 * 2049)]


_lib = None


def load_library() -> C.CDLL:
    """Loads libngs_cuda.so; raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(the ngs-cuda engine has no CPU fallback)")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    P, u8p, u64p, u32p = C.c_void_p, C.POINTER(C.c_uint8), C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)
    lib.ngsq_version.restype = C.c_int
    lib.ngsq_last_error.restype = C.c_char_p
    lib.ngsq_last_error.argtypes = [P]
    lib.ngsq_create.argtypes = [C.c_int, C.POINTER(Config), C.POINTER(P)]
    lib.ngsq_destroy.argtypes = [P]
    lib.ngsq_destroy.restype = None
    lib.ngsq_reset.argtypes = [P]
    lib.ngsq_set_references.argtypes = [P, C.c_uint32, u32p, u8p]
    lib.ngsq_set_range.argtypes = [P, C.c_uint64, C.c_uint64]
    lib.ngsq_bgzf_walk.argtypes = [P, C.c_size_t, C.c_uint64, C.POINTER(Block), C.c_uint32, u32p, C.POINTER(C.c_size_t)]
    lib.ngsq_submit.argtypes = [P, P, C.c_size_t, C.c_uint64]
    lib.ngsq_submit_device.argtypes = [P, P, C.c_size_t, C.POINTER(Block), C.c_uint32]
    lib.ngsq_finish.argtypes = [P]
    lib.ngsq_get_general.argtypes = [P, u64p]
    lib.ngsq_get_tlen.argtypes = [P, u64p, u64p, u64p]
    lib.ngsq_get_gc.argtypes = [P, u64p, u64p, u64p]
    lib.ngsq_get_quality.argtypes = [P, u64p, C.c_size_t, u32p]
    lib.ngsq_get_coverage_contig.argtypes = [P, C.c_uint32, C.POINTER(CovInts), u64p, C.c_size_t]
    lib.ngsq_get_coverage_global.argtypes = [P, u64p]
    lib.ngsq_get_stats.argtypes = [P, C.POINTER(Stats)]
    lib.ngsq_nccl_unique_id.argtypes = [C.c_char_p]
    lib.ngsq_comm_init.argtypes = [P, C.c_int, C.c_int, C.c_char_p]
    lib.ngsq_reduce.argtypes = [P, C.c_int]
    lib.ngsq_set_quality_positions.argtypes = [P, C.c_uint32]
    lib.ngsq_result_buffer.argtypes = [P, C.POINTER(P), C.POINTER(C.c_size_t)]
    lib.ngsq_refresh_results.argtypes = [P]
    lib.ngsq_host_alloc.argtypes = [C.c_size_t]
    lib.ngsq_host_alloc.restype = P
    lib.ngsq_host_free.argtypes = [P]
    lib.ngsq_host_free.restype = None
    lib.ngsq_inflate_to_host.argtypes = [P, P, C.c_size_t, P, C.c_size_t, C.POINTER(C.c_size_t)]
    lib.ngsq_set_reference_bases.argtypes = [P, C.c_uint32, P, C.c_uint64]
    lib.ngsq_get_edits.argtypes = [P, u64p, u64p, u64p, u64p]
    lib.ngsq_get_edit_positions.argtypes = [P, C.c_uint32, u32p, u32p, C.c_uint64]
    lib.ngsq_set_feature_model.argtypes = [P, u8p, u8p]
    lib.ngsq_set_features.argtypes = [P, C.c_uint32, C.c_uint32, u32p, u32p, u8p]
    lib.ngsq_get_features.argtypes = [P, u64p]
    lib.ngsq_wait_copied.argtypes = [P, C.c_uint32]
    lib.ngsq_flush.argtypes = [P]
    lib.ngsq_progress.argtypes = [P, u64p]
    lib.ngsq_host_register.argtypes = [P, C.c_size_t]
    lib.ngsq_host_unregister.argtypes = [P]
    lib.ngsq_get_bai.argtypes = [P, P, C.c_size_t, C.POINTER(C.c_size_t)]
    lib.ngsq_split_reference.argtypes = [P, C.c_uint32]
    lib.ngsq_split_arrays.argtypes = [P, C.c_uint32, C.POINTER(SplitArrays)]
    lib.ngsq_resolve_split.argtypes = [P, C.c_int]
    lib.ngsq_find_record.argtypes = [P, P, C.c_size_t, C.c_uint64, u64p, C.POINTER(C.c_int32)]
    lib.ngsq_join_bai.argtypes = [C.POINTER(P), C.c_uint32, P, C.c_size_t, C.POINTER(C.c_size_t)]
    lib.ngsq_set_index_binning.argtypes = [P, C.c_uint32, C.c_uint32]
    lib.ngsq_get_csi.argtypes = [P, P, C.c_size_t, C.POINTER(C.c_size_t)]
    lib.ngsq_join_csi.argtypes = [C.POINTER(P), C.c_uint32, P, C.c_size_t, C.POINTER(C.c_size_t)]
    _lib = lib
    return lib


def bgzf_walk(data: np.ndarray, file_off: int = 0):
    """K1 on the host: block descriptors for whole blocks in `data` (uint8 array).
    Returns (Block array, n_blocks, bytes consumed)."""
    lib = load_library()
    n = C.c_uint32(0)
    used = C.c_size_t(0)
    rc = lib.ngsq_bgzf_walk(data.ctypes.data, data.size, file_off, None, 0, C.byref(n), C.byref(used))
    if rc:
        raise NgsqError(rc, "malformed BGZF framing")
    arr = (Block * max(n.value, 1))()
    rc = lib.ngsq_bgzf_walk(data.ctypes.data, data.size, file_off, arr, n.value, C.byref(n), C.byref(used))
    if rc:
        raise NgsqError(rc, "malformed BGZF framing")
    return arr, n.value, used.value


@dataclass
class CoverageContig:
    touched: bool
    pileup_too_large: int
    hist: np.ndarray      # 2049 x u64
    bin_sums: np.ndarray  # n_bins x u64


class Engine:
    """One engine = one GPU.  Thin, explicit mirror of the C ABI."""

    def __init__(self, device: int = 0, flags: int = NGSQ_F_RECORD_FACETS | NGSQ_F_COVERAGE, gc_seed: int = 0,
                 max_records: int = 0, reserve_compressed: int = 0, reserve_inflated: int = 0, reserve_blocks: int = 0,
                 launch_blocks: int = 0, quality_positions: int = 0, carry_bytes: int = 0, comp_ring_bytes: int = 0):
        self.lib = load_library()
        cfg = Config(C.sizeof(Config), flags, gc_seed, max_records, reserve_compressed, reserve_inflated, reserve_blocks,
                     launch_blocks, quality_positions, carry_bytes, comp_ring_bytes)
        h = C.c_void_p()
        rc = self.lib.ngsq_create(device, C.byref(cfg), C.byref(h))
        if rc:
            raise NgsqError(rc, self.lib.ngsq_last_error(None).decode())
        self.h = h
        self.n_ref = 0
        self._keep = []  # host buffers that must outlive the run

    def _check(self, rc: int):
        if rc:
            raise NgsqError(rc, self.lib.ngsq_last_error(self.h).decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.ngsq_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self):
        self._check(self.lib.ngsq_reset(self.h))
        self._keep.clear()

    def set_references(self, ref_len, coverage_enabled):
        rl = np.ascontiguousarray(ref_len, dtype=np.uint32)
        ce = np.ascontiguousarray(coverage_enabled, dtype=np.uint8)
        self.n_ref = rl.size
        self._check(self.lib.ngsq_set_references(self.h, rl.size, rl.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                 ce.ctypes.data_as(C.POINTER(C.c_uint8))))

    def set_range(self, first_rec_voffset: int, end_voffset: int = 0):
        self._check(self.lib.ngsq_set_range(self.h, first_rec_voffset, end_voffset))

    def submit(self, data: np.ndarray, file_off: int = 0):
        """data: uint8 numpy array of whole BGZF blocks (host memory, ideally pinned)."""
        self._keep.append(data)
        self._check(self.lib.ngsq_submit(self.h, data.ctypes.data, data.size, file_off))

    def submit_ptr(self, addr: int, nbytes: int, file_off: int = 0):
        self._check(self.lib.ngsq_submit(self.h, addr, nbytes, file_off))

    def flush(self):
        self._check(self.lib.ngsq_flush(self.h))

    def progress(self) -> int:
        v = C.c_uint64(0)
        self._check(self.lib.ngsq_progress(self.h, C.byref(v)))
        return v.value

    def wait_copied(self, submit_index: int):
        self._check(self.lib.ngsq_wait_copied(self.h, submit_index))

    def submit_device(self, dev_ptr: int, nbytes: int, blocks, n_blocks: int):
        self._check(self.lib.ngsq_submit_device(self.h, dev_ptr, nbytes, blocks, n_blocks))

    def finish(self):
        self._check(self.lib.ngsq_finish(self.h))

    def inflate_to_host(self, data: np.ndarray) -> np.ndarray:
        n = C.c_size_t(0)
        # a BGZF block inflates to at most 64 KiB whatever its compressed size (a pile-up of identical records compresses 1000:1)
        _, n_blocks, _ = bgzf_walk(data)
        cap = (int(n_blocks) + 1) * 65536
        out = np.empty(cap, dtype=np.uint8)
        self._check(self.lib.ngsq_inflate_to_host(self.h, data.ctypes.data, data.size, out.ctypes.data, cap, C.byref(n)))
        return out[: n.value].copy()

    # ---- integer getters ----
    def general(self) -> np.ndarray:
        out = np.zeros(34, dtype=np.uint64)
        self._check(self.lib.ngsq_get_general(self.h, out.ctypes.data_as(C.POINTER(C.c_uint64))))
        return out

    def tlen(self):
        hist = np.zeros(1025, dtype=np.uint64)
        p, i = C.c_uint64(0), C.c_uint64(0)
        self._check(self.lib.ngsq_get_tlen(self.h, hist.ctypes.data_as(C.POINTER(C.c_uint64)), C.byref(p), C.byref(i)))
        return hist, p.value, i.value

    def gc(self):
        hist = np.zeros(101, dtype=np.uint64)
        nuc = np.zeros(3, dtype=np.uint64)
        rec = np.zeros(3, dtype=np.uint64)
        u64p = C.POINTER(C.c_uint64)
        self._check(self.lib.ngsq_get_gc(self.h, hist.ctypes.data_as(u64p), nuc.ctypes.data_as(u64p), rec.ctypes.data_as(u64p)))
        return hist, nuc, rec

    def quality(self) -> np.ndarray:
        n = C.c_uint32(0)
        self._check(self.lib.ngsq_get_quality(self.h, None, 0, C.byref(n)))
        out = np.zeros((max(n.value, 1), 94), dtype=np.uint64)
        self._check(self.lib.ngsq_get_quality(self.h, out.ctypes.data_as(C.POINTER(C.c_uint64)), out.shape[0], C.byref(n)))
        return out[: n.value]

    def coverage_contig(self, ref: int, ref_len: int) -> CoverageContig:
        ci = CovInts()
        cap = ref_len // 50000 + 3
        bins = np.zeros(cap, dtype=np.uint64)
        self._check(self.lib.ngsq_get_coverage_contig(self.h, ref, C.byref(ci), bins.ctypes.data_as(C.POINTER(C.c_uint64)), cap))
        return CoverageContig(bool(ci.touched), int(ci.pileup_too_large), np.ctypeslib.as_array(ci.hist).copy(), bins[: ci.n_bins].copy())

    def nonsensical_records(self) -> int:
        v = C.c_uint64(0)
        self._check(self.lib.ngsq_get_coverage_global(self.h, C.byref(v)))
        return v.value

    # ---- Edits (NGSQ_F_EDITS) ----
    def set_reference_bases(self, ref: int, letters):
        """letters: the FASTA sequence of reference `ref` (bytes / uint8 array, line ends removed)."""
        a = np.frombuffer(letters, dtype=np.uint8) if isinstance(letters, (bytes, bytearray)) else np.ascontiguousarray(letters, dtype=np.uint8)
        self._check(self.lib.ngsq_set_reference_bases(self.h, ref, a.ctypes.data, a.size))

    def edits(self):
        """(read_one[513], read_two[513], vaf[101], records stepped through)."""
        one, two, vaf = np.zeros(513, dtype=np.uint64), np.zeros(513, dtype=np.uint64), np.zeros(101, dtype=np.uint64)
        n = C.c_uint64(0)
        u64p = C.POINTER(C.c_uint64)
        self._check(self.lib.ngsq_get_edits(self.h, one.ctypes.data_as(u64p), two.ctypes.data_as(u64p), vaf.ctypes.data_as(u64p), C.byref(n)))
        return one, two, vaf, n.value

    def edit_positions(self, ref: int, length: int):
        """(refs[length + 1], alts[length + 1]) of header sequence `ref`, indexed by 1-based position (the VAF file's input)."""
        refs, alts = np.zeros(length + 1, dtype=np.uint32), np.zeros(length + 1, dtype=np.uint32)
        u32p = C.POINTER(C.c_uint32)
        self._check(self.lib.ngsq_get_edit_positions(self.h, ref, refs.ctypes.data_as(u32p), alts.ctypes.data_as(u32p), length + 1))
        return refs, alts

    # ---- Genomic Features (NGSQ_F_FEATURES) ----
    def set_feature_model(self, names, primary):
        """names: the five configured feature names (5' UTR, 3' UTR, CDS, exon, gene); returns slot_class."""
        sc = np.array([min(i for i in range(5) if names[i] == names[j]) for j in range(5)], dtype=np.uint8)
        pr = np.ascontiguousarray(primary, dtype=np.uint8)
        u8p = C.POINTER(C.c_uint8)
        self._check(self.lib.ngsq_set_feature_model(self.h, sc.ctypes.data_as(u8p), pr.ctypes.data_as(u8p)))
        return sc

    def set_features(self, ref: int, start, stop, cls):
        a, b = np.ascontiguousarray(start, dtype=np.uint32), np.ascontiguousarray(stop, dtype=np.uint32)
        k = np.ascontiguousarray(cls, dtype=np.uint8)
        u32p = C.POINTER(C.c_uint32)
        self._check(self.lib.ngsq_set_features(self.h, ref, a.size, a.ctypes.data_as(u32p), b.ctypes.data_as(u32p), k.ctypes.data_as(C.POINTER(C.c_uint8))))

    def features(self) -> np.ndarray:
        out = np.zeros(9, dtype=np.uint64)
        self._check(self.lib.ngsq_get_features(self.h, out.ctypes.data_as(C.POINTER(C.c_uint64))))
        return out

    # ---- BAI (NGSQ_F_INDEX) ----
    def bai(self) -> bytes:
        """The .bai file of the records submitted since set_range (after finish)."""
        return self._index_bytes(self.lib.ngsq_get_bai)

    # ---- CSI (NGSQ_F_INDEX | NGSQ_F_INDEX_CSI) ----
    def set_index_binning(self, min_shift: int = 14, depth: int = 0):
        """The CSI's binning (depth 0: samtools' rule from the longest reference); before set_references."""
        self._check(self.lib.ngsq_set_index_binning(self.h, min_shift, depth))

    def csi(self) -> bytes:
        """The uncompressed .csi payload of the records submitted since set_range (after finish); the file is its BGZF."""
        return self._index_bytes(self.lib.ngsq_get_csi)

    def _index_bytes(self, getter) -> bytes:
        n = C.c_size_t(0)
        self._check(getter(self.h, None, 0, C.byref(n)))
        buf = np.empty(max(n.value, 1), dtype=np.uint8)
        self._check(getter(self.h, buf.ctypes.data, n.value, C.byref(n)))
        return buf[: n.value].tobytes()

    def find_record(self, data: np.ndarray, file_off: int = 0):
        """Record anchor in whole BGZF blocks `data` (uint8 array) that start at file offset `file_off`: (virtual offset of
        the first offset that starts a chain of plausible records to the end of the window, its reference id), or (0, -1)
        when the window holds none.  Speculative: a range that ends there proves it (ngsq_find_record)."""
        v, r = C.c_uint64(0), C.c_int32(-1)
        self._check(self.lib.ngsq_find_record(self.h, data.ctypes.data, data.size, file_off, C.byref(v), C.byref(r)))
        return v.value, r.value

    def stats(self) -> dict:
        st = Stats()
        self._check(self.lib.ngsq_get_stats(self.h, C.byref(st)))
        return st.as_dict()

    # ---- multi-GPU ----
    def result_buffer(self):
        p = C.c_void_p()
        n = C.c_size_t(0)
        self._check(self.lib.ngsq_result_buffer(self.h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def set_quality_positions(self, n: int):
        self._check(self.lib.ngsq_set_quality_positions(self.h, n))

    def refresh_results(self):
        self._check(self.lib.ngsq_refresh_results(self.h))

    def comm_init(self, n_ranks: int, rank: int, unique_id: bytes):
        self._check(self.lib.ngsq_comm_init(self.h, n_ranks, rank, unique_id))

    def reduce(self, root: int = 0):
        self._check(self.lib.ngsq_reduce(self.h, root))

    # ---- shards cut inside a contig ----
    def split_reference(self, ref: int):
        """Declares reference `ref` split between shards (same set on every engine; before the first submit)."""
        self._check(self.lib.ngsq_split_reference(self.h, ref))

    def split_arrays(self, ref: int) -> dict:
        """Device pointers and lengths of a split reference's partial arrays (for a caller's own collective):
        diff / n_diff (int32), tile_sums / n_tiles (int32), touched (one u64), edit_refs / edit_alts / n_positions (u32);
        a pointer is None when its facet is off."""
        out = SplitArrays()
        self._check(self.lib.ngsq_split_arrays(self.h, ref, C.byref(out)))
        return out.as_dict()

    def resolve_split(self, is_root: bool):
        """After the split arrays were summed into the root's: resolve them there, zero them elsewhere."""
        self._check(self.lib.ngsq_resolve_split(self.h, int(bool(is_root))))


def join_bai(parts) -> bytes:
    """The .bai of a file from its NGSQ_F_INDEX_PART engines, in file order (ngsq_join_bai)."""
    return _join(load_library().ngsq_join_bai, parts)


def join_csi(parts) -> bytes:
    """The uncompressed .csi of a file from its NGSQ_F_INDEX_PART | NGSQ_F_INDEX_CSI engines, in file order (ngsq_join_csi)."""
    return _join(load_library().ngsq_join_csi, parts)


def _join(fn, parts) -> bytes:
    lib = load_library()
    hs = (C.c_void_p * len(parts))(*[p.h.value for p in parts])
    n = C.c_size_t(0)

    def check(rc):
        if rc:
            raise NgsqError(rc, lib.ngsq_last_error(parts[0].h if parts else None).decode())
    check(fn(hs, len(parts), None, 0, C.byref(n)))
    buf = np.empty(max(n.value, 1), dtype=np.uint8)
    check(fn(hs, len(parts), buf.ctypes.data, n.value, C.byref(n)))
    return buf[: n.value].tobytes()


def nccl_unique_id() -> bytes:
    lib = load_library()
    buf = C.create_string_buffer(128)
    rc = lib.ngsq_nccl_unique_id(buf)
    if rc:
        raise NgsqError(rc, lib.ngsq_last_error(None).decode())
    return buf.raw


# ---------------------------------------------------------------- synthetic data
class SynthInfo(C.Structure):
    _fields_ = [("n_records", C.c_uint64), ("inflated_bytes", C.c_uint64), ("header_bytes", C.c_uint64),
                ("bam_bytes", C.c_uint64), ("bai_bytes", C.c_uint64), ("n_blocks", C.c_uint32), ("n_ref", C.c_uint32)]


_synth = None


def synth_layout(shape: int, n_records: int):
    """Records per contig and in the unplaced tail of the logical synthetic file."""
    _load_synth()
    per = (C.c_uint64 * 64)()
    n_ref, tail = C.c_uint32(0), C.c_uint64(0)
    _synth.synth_layout(shape, n_records, per, 64, C.byref(n_ref), C.byref(tail))
    return [per[i] for i in range(n_ref.value)], tail.value


def _load_synth():
    global _synth
    if _synth is None:
        if not os.path.exists(SYNTH_PATH):
            raise ImportError(f"{SYNTH_PATH} is not built: run __graft_entry__.build()")
        _synth = C.CDLL(SYNTH_PATH)
        _synth.synth_bam.argtypes = [C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.POINTER(C.c_void_p),
                                     C.POINTER(C.c_void_p), C.POINTER(SynthInfo)]
        _synth.synth_bam_subset.argtypes = [C.c_int, C.c_uint64, C.c_uint64, C.c_int, C.c_int, C.c_uint64, C.c_int,
                                            C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(SynthInfo)]
        _synth.synth_layout.argtypes = [C.c_int, C.c_uint64, C.POINTER(C.c_uint64), C.c_uint32, C.POINTER(C.c_uint32),
                                        C.POINTER(C.c_uint64)]
        _synth.synth_free.argtypes = [C.c_void_p]
        _synth.synth_free.restype = None


def synth_bam(shape: int, n_records: int, seed: int | None = None, level: int = 6, threads: int = 0,
              contig_mask: int | None = None, with_tail: bool = True):
    """Deterministic synthetic BAM + BAI (tools/bamgen.cpp).  Returns (bam u8 array, bai u8 array, info dict).
    With contig_mask, only those contigs (and the tail if with_tail) of the logical n_records file are written."""
    global _synth
    _load_synth()
    if seed is None:
        seed = 0x5EED0001 + shape
    bam, bai, info = C.c_void_p(), C.c_void_p(), SynthInfo()
    if contig_mask is None:
        rc = _synth.synth_bam(shape, n_records, seed, level, threads, C.byref(bam), C.byref(bai), C.byref(info))
    else:
        rc = _synth.synth_bam_subset(shape, n_records, seed, level, threads, contig_mask, int(with_tail), C.byref(bam),
                                     C.byref(bai), C.byref(info))
    if rc:
        raise RuntimeError(f"synth_bam failed ({rc})")
    # zero-copy views over the malloc'd buffers; freed when the arrays are garbage collected
    a = np.ctypeslib.as_array(C.cast(bam, C.POINTER(C.c_uint8)), shape=(info.bam_bytes,))
    b = np.ctypeslib.as_array(C.cast(bai, C.POINTER(C.c_uint8)), shape=(info.bai_bytes,)).copy()
    _synth.synth_free(bai)
    holder = _MallocHolder(bam.value)
    a = a.view(_OwnedArray)
    a._holder = holder
    return a, b, {n: getattr(info, n) for n, _ in info._fields_}


class _MallocHolder:
    def __init__(self, ptr):
        self.ptr = ptr

    def __del__(self):
        if self.ptr and _synth is not None:
            _synth.synth_free(self.ptr)
            self.ptr = None


class _OwnedArray(np.ndarray):
    """ndarray view that keeps the malloc'd buffer alive (views inherit the holder)."""

    def __array_finalize__(self, obj):
        self._holder = getattr(obj, "_holder", None)
