"""BAI test helpers: the BAI oracle (tests/cpp/bai_oracle.c: oracle_build_bai, oracle_bai_keys) through ctypes, the
micro-BAMs whose indexes the oracle, the writers and the engine must agree on, and a standard BAI region query."""
import bisect
import ctypes as C
import os
import shutil
import struct
import subprocess
import tempfile

import numpy as np

from bamutil import rec, record, reg2bin, write_bam
from helpers import OracleError

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_bai_lib = None


def _lib():
    """The BAI oracle, compiled on first use into a temporary directory (it is test infrastructure, not part of the build)."""
    global _bai_lib
    if _bai_lib is None:
        d = tempfile.mkdtemp(prefix="bai_oracle_")
        try:
            so = os.path.join(d, "libbai_oracle.so")
            subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-std=c11", "-o", so,
                            os.path.join(ROOT, "tests", "cpp", "bai_oracle.c"), "-lz", "-lm"], check=True)
            lib = C.CDLL(so)
        finally:
            shutil.rmtree(d, ignore_errors=True)  # the loaded library stays mapped
        P = C.c_void_p
        lib.oracle_build_bai.argtypes = [P, C.c_size_t, P, C.c_size_t, C.POINTER(C.c_size_t)]
        lib.oracle_bai_keys.argtypes = [P, C.c_size_t, P, C.c_size_t, C.POINTER(C.c_size_t)]
        lib.oracle_last_error.restype = C.c_char_p
        _bai_lib = lib
    return _bai_lib


def _u8(bam):
    return np.ascontiguousarray(np.frombuffer(bam, dtype=np.uint8) if isinstance(bam, (bytes, bytearray)) else bam)


def oracle_bai(bam) -> bytes:
    """The oracle's .bai of a whole BAM (raises OracleError where the reference's `ngs index` would fail)."""
    lib, a = _lib(), _u8(bam)
    cap = max(1 << 20, a.size // 8)
    while True:
        out = np.empty(cap, dtype=np.uint8)
        n = C.c_size_t(0)
        if lib.oracle_build_bai(a.ctypes.data, a.size, out.ctypes.data, cap, C.byref(n)):
            raise OracleError(lib.oracle_last_error().decode())
        if n.value <= cap:
            return out[: n.value].tobytes()
        cap = n.value


KEY_FIELDS = ("ref", "pos", "bin", "beg", "end", "placed", "unmapped", "voff")


def oracle_keys(bam):
    """(list of per-record key tuples in KEY_FIELDS order, error message or None at the first rejected record)."""
    lib, a = _lib(), _u8(bam)
    cap = a.size // 8 + 64
    out = np.zeros((cap, 8), dtype=np.int64)
    n = C.c_size_t(0)
    rc = lib.oracle_bai_keys(a.ctypes.data, a.size, out.ctypes.data, cap, C.byref(n))
    assert n.value <= cap
    keys = [tuple(int(x) for x in row) for row in out[: n.value]]
    return keys, (lib.oracle_last_error().decode() if rc else None)


# ---------------------------------------------------------------- micro-BAMs
REFS = [("chr1", 1 << 27), ("chr2", 100000), ("chr3", 50000), ("chrM", 16390)]


def _m(pos, cigar="100M", ref=0, flag=0, name="r", seq_len=20):
    return rec(name=name, flag=flag, ref=ref, pos=pos, cigar=cigar, seq="ACGT" * (seq_len // 4))


def micro_bams():
    """name -> (bam bytes, bamutil.write_bam's bai bytes): the shapes each rule of the index contract meets."""
    out = {}
    # records that start at offset 0 of a block: every payload is a whole number of records
    recs = [_m(p, name=f"a{i:03d}") for i, p in enumerate([10, 200, 16000, 16500, 20000, 40000, 40001, 900000])]
    size = len(recs[0][0])
    out["block_starts"] = write_bam(REFS, recs, block_payload=[size, 2 * size, size, 3 * size])
    # records that straddle blocks (payloads shorter than a record)
    recs = [_m(p, name=f"b{i:03d}", cigar=c) for i, (p, c) in enumerate([(5, "30M"), (16370, "30M"), (16400, "10M5D10M"),
                                                                         (70000, "50M2N50M"), (131000, "200M")])]
    out["spanning"] = write_bam(REFS, recs, block_payload=37)
    # placed unmapped records without a CIGAR (span 0 -> 1) at multiples of 16384, among mapped ones
    recs = []
    for k in range(6):
        recs.append(_m(16384 * k, cigar="*", flag=0x4, name=f"u{k}"))
        recs.append(_m(16384 * k + 7, name=f"m{k}"))
    out["zero_span_unmapped"] = write_bam(REFS, recs, block_payload=[300, 0xFF00])
    # a record in bin 0: an N skip across the 2^26 boundary
    recs = [_m((1 << 26) - 5000, name="x0"), _m((1 << 26) - 100, cigar="50M1000N50M", name="bin0"), _m((1 << 26) + 10, name="x1")]
    out["bin0"] = write_bam(REFS, recs)
    # a contig with no records between two that have some, then an unplaced tail
    recs = [_m(100 + 50 * i, name=f"c{i}") for i in range(5)] + [_m(300 + 70 * i, ref=2, name=f"e{i}") for i in range(5)]
    recs += [rec(name=f"t{i}", flag=0x4, seq="ACGT") for i in range(3)]
    out["empty_middle"] = write_bam(REFS, recs, block_payload=[200, 150])
    # nothing but unplaced records
    out["unplaced_tail"] = write_bam(REFS, [rec(name=f"t{i}", flag=0x4, seq="ACGTA") for i in range(4)])
    out["header_only"] = write_bam(REFS, [])
    # a read overhanging chrM (16390 bp, windows 0..1) into windows 2 and 3 past its table
    recs = [_m(10, ref=3, name="m0"), _m(16300, ref=3, cigar="40000M", name="over"), _m(16380, ref=3, cigar="5M", name="m1")]
    out["overhang"] = write_bam(REFS, recs, block_payload=[150, 0xFF00])
    return out


def placed_minus_one_bam():
    """An unmapped record with refID 0 and pos -1 before a placed one on the same reference, with its hand-derived index:
    the pos = -1 record is in no bin and counts toward n_no_coor (write_bam would bin it)."""
    a = rec(name="p", flag=0x4, ref=0, pos=-1, seq="ACGT")
    b = _m(100, cigar="10M", name="q")
    bam, _ = write_bam(REFS, [a, b])
    blocks = bgzf_offsets(bam)
    coff = blocks[1][0]  # header block, then the one block of records
    va, vb = coff << 16, (coff << 16) | len(a[0])
    v_end = blocks[2][0] << 16  # EOF block
    bai = b"BAI\x01" + struct.pack("<i", len(REFS))
    bai += struct.pack("<i", 2) + struct.pack("<Ii", reg2bin(100, 110), 1) + struct.pack("<QQ", vb, v_end)
    bai += struct.pack("<IiQQQQ", 37450, 2, vb, v_end, 1, 0) + struct.pack("<i", 1) + struct.pack("<Q", vb)
    bai += struct.pack("<ii", 0, 0) * (len(REFS) - 1) + struct.pack("<Q", 1)
    assert va < vb
    return bam, bai


def bad_record_bams():
    """name -> BAM whose one record the reference's reader or indexer rejects."""
    out = {}
    raw, info = _m(100, cigar="10M", name="badop")
    cig = 4 + 32 + len("badop") + 1
    raw = bytearray(raw)
    raw[cig:cig + 4] = struct.pack("<I", (10 << 4) | 9)
    out["cigar_op"] = write_bam(REFS, [(bytes(raw), info)])[0]
    raw, info = _m(100, name="far")
    raw = bytearray(raw)
    raw[4:8] = struct.pack("<i", len(REFS))  # a reference id the header does not have
    out["ref_id"] = write_bam(REFS, [(bytes(raw), info)])[0]
    raw = bytearray(record(name="over", ref=0, pos=5, cigar="10M", seq="ACGT"))
    raw[4 + 16:4 + 20] = struct.pack("<I", 400)  # l_seq past the end of the record
    out["overrun"] = write_bam(REFS, [(bytes(raw), dict(ref=0, pos=5, span=10, flag=0))])[0]
    out["too_long"] = write_bam([("big", (1 << 29) - 1)], [_m((1 << 29) - 5, ref=0, cigar="10M", name="end")])[0]
    return out


def unsorted_bams():
    """name -> (BAM, index of the first record out of order)."""
    return {
        "position": (write_bam(REFS, [_m(500, name="a"), _m(400, name="b"), _m(600, name="c")])[0], 1),
        "reference": (write_bam(REFS, [_m(500, ref=1, name="a"), _m(400, ref=0, name="b")])[0], 1),
        "after_unplaced": (write_bam(REFS, [_m(500, name="a"), rec(name="u", flag=4, seq="AC"), _m(600, name="c")])[0], 2),
    }


# ---------------------------------------------------------------- BGZF / query
def bgzf_offsets(bam):
    """[(coffset, inflated start, isize)] of every block, empty ones included."""
    out, o, at = [], 0, 0
    b = bytes(bam)
    while o < len(b):
        total = struct.unpack_from("<H", b, o + 16)[0] + 1
        isize = struct.unpack_from("<I", b, o + total - 4)[0]
        out.append((o, at, isize))
        at += isize
        o += total
    return out


def region_query(bai_bytes, bam, keys, ref, beg, end):
    """Records a standard BAI query of [beg, end) on `ref` returns, filtered by overlap: indices into `keys`."""
    from ngs_b200.formats import parse_bai
    bai = parse_bai(bai_bytes)
    R = bai.refs[ref]
    blocks = bgzf_offsets(bam)
    start_of = {c: s for c, s, _ in blocks}
    to_stream = lambda v: start_of[v >> 16] + (v & 0xFFFF)  # noqa: E731
    rec_stream = [to_stream(k[7]) for k in keys]  # file order: ascending
    bins = reg2bins(beg, end)
    min_off = R.linear[beg >> 14] if (beg >> 14) < len(R.linear) else (R.linear[-1] if R.linear else 0)
    hit = set()
    for b, chunks in R.bins.items():
        if b not in bins:
            continue
        for cb, ce in chunks:
            if ce <= min_off:
                continue
            lo, hi = to_stream(cb), to_stream(ce)
            for i in range(bisect.bisect_left(rec_stream, lo), bisect.bisect_left(rec_stream, hi)):
                k = keys[i]
                if k[5] and k[0] == ref and k[3] < end and k[4] > beg:
                    hit.add(i)
    return hit


def reg2bins(beg, end):
    """SAM spec 5.3: every bin that may hold a record overlapping [beg, end)."""
    end -= 1
    out = {0}
    for first, shift in ((1, 26), (9, 23), (73, 20), (585, 17), (4681, 14)):
        out.update(range(first + (beg >> shift), first + (end >> shift) + 1))
    return out


def brute_force(keys, ref, beg, end):
    return {i for i, k in enumerate(keys) if k[5] and k[0] == ref and k[3] < end and k[4] > beg}

