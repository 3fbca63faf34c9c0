"""Host-side format helpers for the harness (tests, bench.py): BAM header, BAI, genome table,
shard planning.  Mirrors what the reference does on the host before its hot loops:
`open_and_parse` (src/utils/formats/bam.rs:77-123), the concordance check
(src/qc/command.rs:258-272), `supports_sequence_name` (coverage.rs:133-138).  The C++ host
driver (ngs_b200/host) holds the same logic for the product path.
"""
from __future__ import annotations

import bisect
import os
import re
import struct
from dataclasses import dataclass, field

import numpy as np

from . import ffi

_HERE = os.path.dirname(os.path.abspath(__file__))


def grch38_no_alt_names() -> dict[str, str]:
    """name -> kind (C chromosome, M mitochondrion, E ebv, L unlocalized, P unplaced), from the
    table shared with the C++ host (reference: utils/genome/ncbi/grch38_no_alt.rs:46-283)."""
    out = {}
    with open(os.path.join(_HERE, "host", "grch38_no_alt_names.inc")) as f:
        for m in re.finditer(r'NGSQ_SEQ\("([^"]+)", \'(.)\'\)', f.read()):
            out[m.group(1)] = m.group(2)
    return out


_GENOME = None


def is_primary(name: str) -> bool:
    """get_primary_assembly membership (utils/genome.rs:59-83): autosomes, sex, unlocalized, unplaced."""
    global _GENOME
    if _GENOME is None:
        _GENOME = grch38_no_alt_names()
    return _GENOME.get(name) in ("C", "L", "P")


def is_known(name: str) -> bool:
    global _GENOME
    if _GENOME is None:
        _GENOME = grch38_no_alt_names()
    return name in _GENOME


@dataclass
class BamHeader:
    text: str
    refs: list  # [(name, length)]
    header_bytes: int       # inflated bytes occupied by the header
    first_voffset: int      # virtual offset of the first record


class NeedMore(Exception):
    pass


def parse_bam_header(buf: bytes):
    """Parses the BAM header from inflated bytes; raises NeedMore if `buf` is too short."""
    def need(n):
        if len(buf) < n:
            raise NeedMore()
    need(12)
    if buf[:4] != b"BAM\x01":
        raise ValueError("not a BAM file (bad magic)")
    l_text = struct.unpack_from("<i", buf, 4)[0]
    o = 8 + l_text
    need(o + 4)
    text = buf[8:o].decode("utf-8", "replace")
    n_ref = struct.unpack_from("<i", buf, o)[0]
    o += 4
    refs = []
    for _ in range(n_ref):
        need(o + 4)
        l_name = struct.unpack_from("<i", buf, o)[0]
        o += 4
        need(o + l_name + 4)
        name = buf[o:o + l_name - 1].decode()
        o += l_name
        l_ref = struct.unpack_from("<i", buf, o)[0]
        o += 4
        refs.append((name, l_ref))
    return text, refs, o


def read_header(engine: ffi.Engine, bam: np.ndarray) -> BamHeader:
    """Header from the first BGZF block(s), inflated ON THE GPU (ngsq_inflate_to_host)."""
    take = 1 << 16
    while True:
        chunk = bam[: min(take, bam.size)]
        blocks, n, used = ffi.bgzf_walk(chunk)
        if n == 0 and chunk.size == bam.size:
            raise ValueError("no BGZF block in file")
        data = engine.inflate_to_host(chunk[:used]) if used else b""
        try:
            text, refs, hlen = parse_bam_header(bytes(data))
        except NeedMore:
            if chunk.size == bam.size:
                raise ValueError("truncated BAM header")
            take *= 4
            continue
        # virtual offset of the byte right after the header
        acc = 0
        voff = None
        for i in range(n):
            b = blocks[i]
            if hlen < acc + b.isize:
                voff = (b.coffset << 16) | (hlen - acc)
                break
            acc += b.isize
        if voff is None:
            # header ends exactly on a block boundary: first record starts the next block
            voff = used << 16
        return BamHeader(text, refs, hlen, voff)


@dataclass
class BaiRef:
    bins: dict = field(default_factory=dict)     # bin -> [(beg, end)]
    linear: list = field(default_factory=list)
    ref_beg: int | None = None                   # pseudo-bin 37450
    ref_end: int | None = None
    n_mapped: int = 0
    n_unmapped: int = 0


@dataclass
class Bai:
    refs: list
    n_no_coor: int | None


def parse_bai(buf: bytes) -> Bai:
    if buf[:4] != b"BAI\x01":
        raise ValueError("bad BAI magic")
    n_ref = struct.unpack_from("<i", buf, 4)[0]
    o = 8
    refs = []
    for _ in range(n_ref):
        r = BaiRef()
        n_bin = struct.unpack_from("<i", buf, o)[0]
        o += 4
        for _ in range(n_bin):
            b, n_chunk = struct.unpack_from("<Ii", buf, o)
            o += 8
            chunks = [struct.unpack_from("<QQ", buf, o + 16 * k) for k in range(n_chunk)]
            o += 16 * n_chunk
            if b == 37450 and n_chunk == 2:
                r.ref_beg, r.ref_end = chunks[0]
                r.n_mapped, r.n_unmapped = chunks[1]
            else:
                r.bins[b] = chunks
        n_intv = struct.unpack_from("<i", buf, o)[0]
        o += 4
        r.linear = list(struct.unpack_from(f"<{n_intv}Q", buf, o))
        o += 8 * n_intv
        refs.append(r)
    n_no_coor = struct.unpack_from("<Q", buf, o)[0] if o + 8 <= len(buf) else None
    return Bai(refs, n_no_coor)


@dataclass
class CsiRef:
    bins: dict = field(default_factory=dict)     # bin -> [(beg, end)]
    loffset: dict = field(default_factory=dict)  # bin -> loffset
    ref_beg: int | None = None                   # pseudo-bin n_bins + 1
    ref_end: int | None = None
    n_mapped: int = 0
    n_unmapped: int = 0


@dataclass
class Csi:
    min_shift: int
    depth: int
    aux: bytes
    refs: list
    n_no_coor: int | None


def parse_csi(buf: bytes) -> Csi:
    """An uncompressed CSIv1 payload (a .csi file after gzip.decompress)."""
    if buf[:4] != b"CSI\x01":
        raise ValueError("bad CSI magic")
    min_shift, depth, l_aux = struct.unpack_from("<iii", buf, 4)
    aux = bytes(buf[16:16 + l_aux])
    o = 16 + l_aux
    n_ref = struct.unpack_from("<i", buf, o)[0]
    o += 4
    meta = ((1 << 3 * (depth + 1)) - 1) // 7 + 1
    refs = []
    for _ in range(n_ref):
        r = CsiRef()
        n_bin = struct.unpack_from("<i", buf, o)[0]
        o += 4
        for _ in range(n_bin):
            b, loff, n_chunk = struct.unpack_from("<IQi", buf, o)
            o += 16
            chunks = [struct.unpack_from("<QQ", buf, o + 16 * k) for k in range(n_chunk)]
            o += 16 * n_chunk
            if b == meta and n_chunk == 2:
                r.ref_beg, r.ref_end = chunks[0]
                r.n_mapped, r.n_unmapped = chunks[1]
            else:
                r.bins[b] = chunks
                r.loffset[b] = loff
        refs.append(r)
    n_no_coor = struct.unpack_from("<Q", buf, o)[0] if o + 8 <= len(buf) else None
    return Csi(min_shift, depth, aux, refs, n_no_coor)


@dataclass
class Shard:
    first_voffset: int   # first record owned
    end_voffset: int     # first record not owned (0 = to EOF)
    contigs: list        # reference ids whose coverage this shard owns


def plan_shards(header: BamHeader, bai: Bai, n_shards: int, file_size: int) -> list:
    """Contig-aligned cuts from the BAI pseudo-bins (SURVEY 8(e)): contiguous runs of contigs
    balanced by compressed bytes, so every coverage position is owned by exactly one shard and the
    only exchange is the final sum-reduce.  The last shard runs to EOF (unplaced-unmapped tail)."""
    spans = []  # (ref, beg_voffset, end_voffset)
    for c, r in enumerate(bai.refs):
        if r.ref_beg is not None and r.ref_end is not None and r.ref_end > r.ref_beg:
            spans.append((c, r.ref_beg, r.ref_end))
    if n_shards <= 1 or not spans:
        return [Shard(header.first_voffset, 0, list(range(len(header.refs))))]
    spans.sort(key=lambda s: s[1])
    total = file_size - (header.first_voffset >> 16)
    shards = []
    start_v = header.first_voffset
    acc_start = header.first_voffset >> 16
    cur = []
    k = 0
    for i, (c, beg, end) in enumerate(spans):
        cur.append(c)
        done_bytes = (end >> 16) - (header.first_voffset >> 16)
        remaining_contigs = len(spans) - i - 1
        remaining_shards = n_shards - len(shards) - 1
        target = total * (len(shards) + 1) / n_shards
        if remaining_shards > 0 and (done_bytes >= target or remaining_contigs <= remaining_shards - 1) and i + 1 < len(spans):
            nxt = spans[i + 1][1]
            shards.append(Shard(start_v, nxt, cur))
            start_v = nxt
            cur = []
    shards.append(Shard(start_v, 0, cur))
    while len(shards) < n_shards:
        shards.append(Shard(0, 0, []))  # empty shard (more GPUs than contigs)
    return shards


def bai_anchors(bai: Bai) -> list:
    """Record starts a shard may be cut at: every contig's first record (pseudo-bin 37450) and its linear-index ioffsets,
    ascending and distinct (zeros, entries below the contig's first record and repeats dropped)."""
    out = set()
    for r in bai.refs:
        if r.ref_beg is None or r.ref_end is None or r.ref_end <= r.ref_beg:
            continue
        out.add(r.ref_beg)
        out.update(v for v in r.linear if v and r.ref_beg <= v < r.ref_end)
    return sorted(out)


def plan_shards_split(header: BamHeader, bai: Bai, n_shards: int, file_size: int):
    """Shards cut inside contigs at BAI anchors, balanced by compressed bytes (mirror of plan_shards_split in
    ngs_b200/host/bam.hpp).  Returns (shards, split): `split` lists the contigs with records on both sides of a cut, in
    ascending order; a shard's `contigs` are the references it holds records of.  Shards past the anchors are empty."""
    first = header.first_voffset
    cand = [v for v in bai_anchors(bai) if v > first]
    base = first >> 16
    total = float(max(file_size - base, 0))
    m = len(cand)
    n_cuts = min(max(n_shards - 1, 0), m)
    key = [(v >> 16) - base for v in cand]
    cuts, lo = [], 0
    for k in range(1, n_cuts + 1):
        target = total * k / n_shards
        hi = m - (n_cuts - k)
        j = bisect.bisect_left(key, target, lo, hi)  # the nearest candidate in [lo, hi), ties: the earlier one
        if j == hi or (j > lo and target - key[j - 1] <= key[j] - target):
            j -= 1
        cuts.append(cand[j])
        lo = j + 1
    bounds = [first] + cuts
    extents = [(c, r.ref_beg, r.ref_end) for c, r in enumerate(bai.refs)
               if r.ref_beg is not None and r.ref_end is not None and r.ref_end > r.ref_beg]
    shards = []
    for i, b in enumerate(bounds):
        end = bounds[i + 1] if i + 1 < len(bounds) else 0
        shards.append(Shard(b, end, [c for c, beg, e in extents if e > b and (end == 0 or beg < end)]))
    split = [c for c, beg, e in extents if any(beg < v < e for v in cuts)]
    while len(shards) < n_shards:
        shards.append(Shard(0, 0, []))
    return shards, split


def shard_byte_range(shard: Shard, blocks, n_blocks: int, file_size: int):
    """Compressed byte range [lo, hi) a shard must submit: from the block holding its first record
    through the block holding end_voffset (its last record may end inside that block)."""
    lo = shard.first_voffset >> 16
    if shard.end_voffset == 0:
        return lo, file_size
    co, uo = shard.end_voffset >> 16, shard.end_voffset & 0xFFFF
    if uo == 0:
        return lo, co
    # include the block at `co`
    for i in range(n_blocks):
        if blocks[i].coffset == co:
            return lo, co + blocks[i].csize
    raise ValueError("end_voffset does not address a BGZF block")
