"""CSI test helpers: the CSI oracle (tests/cpp/csi_oracle.c: oracle_build_csi, oracle_csi_keys, oracle_csi_default_depth)
through ctypes, htslib's CSI region query, and BAMs over references a BAI cannot address.  The micro-BAMs, the BGZF walk and
the brute-force query are baiutil's."""
import bisect
import ctypes as C
import os
import shutil
import struct
import subprocess
import tempfile

import numpy as np

from baiutil import _m, _u8, bgzf_offsets
from bamutil import rec, write_bam
from helpers import OracleError

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_csi_lib = None


def _lib():
    """The CSI oracle, compiled on first use into a temporary directory (it is test infrastructure, not part of the build)."""
    global _csi_lib
    if _csi_lib is None:
        d = tempfile.mkdtemp(prefix="csi_oracle_")
        try:
            so = os.path.join(d, "libcsi_oracle.so")
            subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-std=c11", "-o", so,
                            os.path.join(ROOT, "tests", "cpp", "csi_oracle.c"), "-lz", "-lm"], check=True)
            lib = C.CDLL(so)
        finally:
            shutil.rmtree(d, ignore_errors=True)  # the loaded library stays mapped
        P = C.c_void_p
        lib.oracle_last_error.restype = C.c_char_p
        lib.oracle_build_csi.argtypes = [P, C.c_size_t, C.c_int, C.c_int, P, C.c_size_t, C.POINTER(C.c_size_t)]
        lib.oracle_csi_keys.argtypes = [P, C.c_size_t, C.c_int, C.c_int, P, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_int)]
        lib.oracle_csi_default_depth.argtypes = [C.c_uint64, C.c_int]
        _csi_lib = lib
    return _csi_lib


def oracle_csi(bam, min_shift=14, depth=0) -> bytes:
    """The oracle's uncompressed .csi payload (depth 0: samtools' rule); raises OracleError where indexing fails."""
    lib, a = _lib(), _u8(bam)
    cap = max(1 << 20, a.size // 8)
    while True:
        out = np.empty(cap, dtype=np.uint8)
        n = C.c_size_t(0)
        if lib.oracle_build_csi(a.ctypes.data, a.size, min_shift, depth, out.ctypes.data, cap, C.byref(n)):
            raise OracleError(lib.oracle_last_error().decode())
        if n.value <= cap:
            return out[: n.value].tobytes()
        cap = n.value


def oracle_csi_keys(bam, min_shift=14, depth=0):
    """(per-record key tuples in KEY_FIELDS order with CSI bins, error message or None, the depth used)."""
    lib, a = _lib(), _u8(bam)
    cap = a.size // 8 + 64
    while True:
        out = np.zeros((cap, 8), dtype=np.int64)
        n, d = C.c_size_t(0), C.c_int(0)
        rc = lib.oracle_csi_keys(a.ctypes.data, a.size, min_shift, depth, out.ctypes.data, cap, C.byref(n), C.byref(d))
        if n.value <= cap:
            break
        cap = n.value
    keys = [tuple(int(x) for x in row) for row in out[: n.value]]
    return keys, (lib.oracle_last_error().decode() if rc else None), d.value


def csi_default_depth(max_len, min_shift=14):
    return _lib().oracle_csi_default_depth(max_len, min_shift)


def csi_reg2bins(beg, end, min_shift, depth):
    """htslib hts_reg2bins: every bin of a CSI that may hold a record overlapping [beg, end)."""
    end -= 1
    out, t, s = set(), 0, min_shift + 3 * depth
    for lv in range(depth + 1):
        out.update(range(t + (beg >> s), t + (end >> s) + 1))
        s -= 3
        t += 1 << 3 * lv
    return out


def csi_min_offset(R, beg, min_shift, depth):
    """htslib's CSI query bound: the loffset of the leaf bin of `beg`, or of the nearest bin to its left (then its parents')
    that the index holds; 0 when there is none."""
    b = ((1 << 3 * depth) - 1) // 7 + (beg >> min_shift)
    while b and b not in R.loffset:
        first = (((b - 1) >> 3) << 3) + 1
        b = b - 1 if b > first else (b - 1) >> 3
    return R.loffset.get(b, 0)


def csi_region_query(csi_bytes, bam, keys, ref, beg, end):
    """Records a standard CSI query of [beg, end) on `ref` returns, filtered by overlap: indices into `keys`."""
    from ngs_b200.formats import parse_csi
    csi = parse_csi(csi_bytes)
    R = csi.refs[ref]
    blocks = bgzf_offsets(bam)
    start_of = {c: s for c, s, _ in blocks}
    to_stream = lambda v: start_of[v >> 16] + (v & 0xFFFF)  # noqa: E731
    rec_stream = [to_stream(k[7]) for k in keys]
    bins = csi_reg2bins(beg, end, csi.min_shift, csi.depth)
    min_off = csi_min_offset(R, beg, csi.min_shift, csi.depth)
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


def _at(pos, cigar="100M", ref=0, flag=0, name="r"):
    """A record at any position: bamutil.record packs the bin field in 16 bits, so a record past 2^29 gets 4680 (no bin)."""
    raw, info = _m(0, cigar=cigar, ref=ref, flag=flag, name=name)
    raw = bytearray(raw)
    raw[8:12] = struct.pack("<i", pos)
    raw[14:16] = struct.pack("<H", 4680)
    info["pos"] = pos
    return bytes(raw), info


def big_reference_bams():
    """name -> BAM over references of 2^29 - 1, 2^29, 2^30 and 2^31 - 1 bases: records on both sides of 2^29, 2^30 and the
    bin boundaries of every level, reads across them (N skips, deletions), zero spans, a read overhanging its reference's end,
    empty references and an unplaced tail."""
    out = {}
    for L in ((1 << 29) - 1, 1 << 29, 1 << 30, (1 << 31) - 1):
        refs = [("big", L), ("empty", 5000), ("tail", L)]
        # every multiple of 2^26, and next to 2^29 and 2^30 the bin boundaries of every smaller level (2^12 .. 2^25)
        cuts = {b for b in range(0, L, 1 << 26)}
        cuts |= {c + k * (1 << s) for c in (1 << 29, 1 << 30) for s in range(12, 26) for k in (-1, 1)}
        cuts = sorted(cuts)
        recs, i = [], 0
        for b in cuts:
            if b >= L:
                continue
            for pos, cig in ((b - 150, "100M"), (b - 60, "100M"), (b - 1, "*"), (b - 30, "10M1000N10M"), (b, "50M"),
                             (b + 5, "20M40000N20M")):
                if 0 <= pos < L:
                    recs.append((pos, cig))
        recs.append((L - 40, "100M"))  # overhangs the end of its reference
        recs.sort()
        rows = [_at(p, cigar=c, name=f"b{i}") for i, (p, c) in enumerate(recs)]
        rows += [_at(p, cigar="30M", ref=2, name=f"t{j}") for j, p in enumerate((10, L // 2, L - 300))]
        rows += [rec(name=f"u{j}", flag=0x4, seq="ACGT") for j in range(2)]
        out[f"len{L}"] = write_bam(refs, rows, block_payload=[500, 0xFF00, 3000])[0]
    return out
