"""Read groups (`qc --cuda-by-read-group`, NGSQ_F_READ_GROUPS) in the tests: the oracle's pass 1 restricted to one group
(tests/cpp/oracle_read_groups.c, which compiles oracle/ngsqc_oracle.c unchanged), an independent Python restatement of
htslib's bam_aux_get rule on top of the Python facet restatement of test_oracle_vs_python.py, hand-built aux blocks, and the
engine's per-group integers."""
import ctypes as C
import os
import struct
import subprocess
import tempfile
from unittest import mock

import numpy as np

from helpers import OracleError

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_lib = None


def rg_oracle_lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="rg_oracle"), "liboracle_rg.so")
        subprocess.run(["gcc", "-O2", "-fPIC", "-shared", "-std=c11", "-ffp-contract=off", "-o", out,
                        os.path.join(ROOT, "tests", "cpp", "oracle_read_groups.c"), "-lz", "-lm"], check=True)
        lib = C.CDLL(out)
        P = C.c_void_p
        lib.oracle_rg_run.restype = P
        lib.oracle_rg_run.argtypes = [P, C.c_size_t, C.c_uint64, C.c_uint64, C.POINTER(C.c_char_p), C.c_uint32, C.c_int64]
        lib.oracle_last_error.restype = C.c_char_p
        lib.oracle_write_json.argtypes = [P, C.c_char_p]
        for name in ["oracle_get_general", "oracle_get_quality"]:
            getattr(lib, name).argtypes = [P, P]
        lib.oracle_get_tlen.argtypes = [P, P, P, P]
        lib.oracle_get_gc.argtypes = [P, P, P, P]
        lib.oracle_quality_positions.restype = C.c_uint64
        lib.oracle_quality_positions.argtypes = [P]
        _lib = lib
    return _lib


def oracle_group_ints(bam, ids, group=-1, n_records=0, gc_seed=0, json_path=None):
    """The four record facets of the records of read group `group` (index into ids; len(ids) = ungrouped; -1 = all)."""
    lib = rg_oracle_lib()
    bam = np.ascontiguousarray(bam)
    arr = (C.c_char_p * max(len(ids), 1))(*[i.encode() if isinstance(i, str) else i for i in ids])
    h = lib.oracle_rg_run(bam.ctypes.data, bam.size, n_records, gc_seed, arr, len(ids), group)
    if not h:
        raise OracleError(lib.oracle_last_error().decode())
    g = np.zeros(34, np.uint64)
    lib.oracle_get_general(h, g.ctypes.data)
    th = np.zeros(1025, np.uint64)
    p, i = C.c_uint64(0), C.c_uint64(0)
    lib.oracle_get_tlen(h, th.ctypes.data, C.addressof(p), C.addressof(i))
    gh, nuc, rec = np.zeros(101, np.uint64), np.zeros(3, np.uint64), np.zeros(3, np.uint64)
    lib.oracle_get_gc(h, gh.ctypes.data, nuc.ctypes.data, rec.ctypes.data)
    nq = lib.oracle_quality_positions(h)
    q = np.zeros((max(nq, 1), 94), np.uint64)
    if nq:
        lib.oracle_get_quality(h, q.ctypes.data)
    if json_path:
        lib.oracle_write_json(h, json_path.encode())
    return dict(general=g, tlen_hist=th, tlen_processed=p.value, tlen_ignored=i.value, gc_hist=gh, gc_nuc=nuc, gc_rec=rec,
                quality=q[:nq])


# ---------------------------------------------------------------- the Python restatement
_SIZES = {"A": 1, "c": 1, "C": 1, "s": 2, "S": 2, "i": 4, "I": 4, "f": 4}


def record_group(b: bytes, ids):
    """htslib's bam_aux_get for RG on a record (bytes without block_size): the index of its ID, len(ids) when ungrouped;
    ValueError for a malformed field in front of the first RG."""
    l_name, n_cig, l_seq = b[8], struct.unpack_from("<H", b, 12)[0], struct.unpack_from("<I", b, 16)[0]
    o = 32 + l_name + 4 * n_cig + (l_seq + 1) // 2 + l_seq
    while o < len(b):
        if len(b) - o < 3:
            raise ValueError("short aux field")
        tag, ty = b[o:o + 2], chr(b[o + 2])
        o += 3
        if tag == b"RG":
            if ty != "Z" or b.find(b"\0", o) < 0:
                return len(ids)
            v = b[o:b.index(b"\0", o)].decode("latin-1")
            return ids.index(v) if v in ids else len(ids)
        if ty in _SIZES:
            n = _SIZES[ty]
        elif ty in "ZH":
            z = b.find(b"\0", o)
            if z < 0:
                raise ValueError("no NUL")
            n = z - o + 1
        elif ty == "B":
            if len(b) - o < 5 or chr(b[o]) not in "cCsSiIf":
                raise ValueError("bad B array")
            n = 5 + struct.unpack_from("<I", b, o + 1)[0] * _SIZES[chr(b[o])]
        else:
            raise ValueError(f"aux type {ty!r}")
        if len(b) - o < n:
            raise ValueError("aux field runs past the record")
        o += n
    return len(ids)


def python_group_ints(raw: bytes, ids, group, gc_seed=0):
    """test_oracle_vs_python's restatement over the records of one group (at their own virtual offsets)."""
    import test_oracle_vs_python as tv
    from ngs_b200 import formats
    refs, recs = tv._records(raw)
    keep = [(v, b) for v, b in recs if group < 0 or record_group(b, ids) == group]
    with mock.patch.object(tv, "_records", lambda _raw: (refs, keep)):
        out = tv._python_facets(raw, gc_seed, formats.is_primary)
    return out


# ---------------------------------------------------------------- hand-built aux blocks
def aux_z(tag, v):
    return tag.encode() + b"Z" + (v.encode("latin-1") if isinstance(v, str) else v) + b"\0"


def aux_h(tag, v):
    return tag.encode() + b"H" + v.encode() + b"\0"


def aux_b(tag, sub, values):
    fmt = {"c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I", "f": "f"}[sub]
    return tag.encode() + b"B" + sub.encode() + struct.pack("<I", len(values)) + struct.pack(f"<{len(values)}{fmt}", *values)


def aux_scalar(tag, ty, v):
    fmt = {"A": "c", "c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I", "f": "f"}[ty]
    return tag.encode() + ty.encode() + struct.pack("<" + fmt, v)


# ---------------------------------------------------------------- the engine
def engine_group_ints(eng, n_groups):
    """[sample, group 0, .., group n_groups (ungrouped)] integer dicts of a finished NGSQ_F_READ_GROUPS engine."""
    from helpers import collect
    out = []
    for g in [-1] + list(range(n_groups + 1)):
        eng.select_read_group(g)
        out.append(collect(eng, [], [], records=True, coverage=False))
    eng.select_read_group(-1)
    return out[0], out[1:]


def sum_groups(groups):
    """Element-wise sum of the groups' integers (the quality length takes the max)."""
    keys = ["general", "tlen_hist", "gc_hist", "gc_nuc", "gc_rec"]
    s = {k: sum(g[k].astype(np.uint64) for g in groups) for k in keys}
    s["tlen_processed"] = sum(g["tlen_processed"] for g in groups)
    s["tlen_ignored"] = sum(g["tlen_ignored"] for g in groups)
    n = max(g["quality"].shape[0] for g in groups)
    q = np.zeros((n, 94), np.uint64)
    for g in groups:
        q[:g["quality"].shape[0]] += g["quality"]
    s["quality"] = q
    return s


def write_rg_bam(refs, records, ids, **kw):
    """bamutil.write_bam with @RG lines for ids in the header."""
    import bamutil
    plain = bamutil.header_bytes

    def with_rg(rs):
        h = plain(rs)
        l_text = struct.unpack_from("<i", h, 4)[0]
        text = h[8:8 + l_text] + "".join(f"@RG\tID:{i}\tSM:s\n" for i in ids).encode()
        return b"BAM\x01" + struct.pack("<i", len(text)) + text + h[8 + l_text:]
    with mock.patch.object(bamutil, "header_bytes", with_rg):
        return bamutil.write_bam(refs, records, **kw)


def adversarial_records(seed=4):
    """Records whose RG sits behind every kind of aux field, RG of other types, two RG tags, undeclared values, the
    rg1 / rg10 prefix pair, no aux block; with the IDs they are meant for."""
    import random
    from bamutil import rec
    rng = random.Random(seed)
    ids = ["rg1", "rg10", "lane 2/x", "r%g"]
    seq = lambda n: "".join(rng.choice("ACGT") for _ in range(n))  # noqa: E731
    fronts = [b"", aux_scalar("XA", "A", b"q"), aux_scalar("Xc", "c", -3), aux_scalar("XC", "C", 200), aux_scalar("Xs", "s", -300),
              aux_scalar("XS", "S", 60000), aux_scalar("Xi", "i", -70000), aux_scalar("XI", "I", 4000000000), aux_scalar("Xf", "f", 1.5),
              aux_z("MM", "C+m?," + ",".join(str(rng.randrange(9)) for _ in range(400))), aux_h("XH", "0A1B" * 200)]
    fronts += [aux_b("XB", sub, vals) for sub, vals in [("c", [-1, 2]), ("C", [1, 255]), ("s", [-2, 3, 4]), ("S", [65535]),
                                                        ("i", [-5] * 7), ("I", [7] * 100), ("f", [0.5, 2.0])]]
    tails = [aux_z("RG", "rg1"), aux_z("RG", "rg10"), aux_z("RG", "rg100"), aux_z("RG", "rg"), aux_z("RG", "lane 2/x"),
             aux_z("RG", "r%g"), aux_scalar("RG", "A", b"r"), aux_scalar("RG", "i", 1), aux_z("RG", "rg10") + aux_z("RG", "rg1"),
             aux_z("rg", "rg1"), b""]
    rs = []
    i = 0
    for front in fronts:
        for tail in tails:
            for k in range(3):
                n = 90 + 7 * ((i + k) % 5)  # 90 .. 118: too short for GC, and windows that start at an offset
                rs.append(rec(name=f"a{i}_{k}", flag=[0x41, 0x81, 0x400, 0x100, 0x63, 0x4 | 0x1 | 0x8][(i + k) % 6], ref=0, pos=100 + 3 * i,
                              mapq=(i * 7) % 60, cigar=f"{n}M", next_ref=0, next_pos=10, tlen=[0, 300, 1024, 1025, -7][(i + k) % 5],
                              seq=seq(n), qual=[rng.randrange(94) for _ in range(n)] if k != 2 else None, aux=front + tail))
            i += 1
    return ids, rs
