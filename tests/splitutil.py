"""The records of one coordinate-sorted BAM S written as several BAM files with S's header (for `qc --cuda-also`): in contiguous
chunks, round-robin (each file sorted, the coordinates of the files interleave, as per-lane files do) or assigned at random.
Each file's records keep S's order; they are packed into BGZF blocks of `block_payload` bytes, as tests/orderutil.py does."""
import struct

import numpy as np

from bamutil import EOF_BLOCK, bgzf_block
from orderutil import split_records

SPLITS = ("contiguous", "round_robin", "random")


def write_file(hdr: bytes, recs, block_payload=0x7100, level=1) -> np.ndarray:
    stream = b"".join(recs)
    out = bytearray(bgzf_block(hdr, level))
    for o in range(0, len(stream), block_payload):
        out += bgzf_block(stream[o:o + block_payload], level)
    out += EOF_BLOCK
    return np.frombuffer(bytes(out), dtype=np.uint8).copy()


def groups_of(n, k, kind, seed=0):
    """Record indices of each of k files."""
    if kind == "contiguous":
        return [list(g) for g in np.array_split(np.arange(n), k)]
    if kind == "round_robin":
        return [list(range(i, n, k)) for i in range(k)]
    if kind == "random":
        a = np.random.default_rng(seed).integers(0, k, n)
        return [list(np.flatnonzero(a == i)) for i in range(k)]
    raise ValueError(kind)


def split_bam(bam, k, kind, seed=0, block_payload=0x7100, level=1):
    """S's records in k files (some may hold no record)."""
    hdr, recs = split_records(bam)
    return [write_file(hdr, [recs[i] for i in g], block_payload, level) for g in groups_of(len(recs), k, kind, seed)]


def flag(r: bytes) -> int:
    return struct.unpack_from("<H", r, 18)[0]


def edge_files(bam, block_payload=0x7100, level=1):
    """S's records as: a header-only file, a file of S's first mapped record, the file of every unmapped record, then the rest
    in two contiguous files."""
    hdr, recs = split_records(bam)
    unmapped = [i for i, r in enumerate(recs) if flag(r) & 4]
    assert unmapped, "S has no unmapped record"
    mapped = [i for i, r in enumerate(recs) if not flag(r) & 4]
    half = (len(mapped) + 1) // 2
    groups = [[], mapped[:1], unmapped, mapped[1:half], mapped[half:]]
    return [write_file(hdr, [recs[i] for i in g], block_payload, level) for g in groups]
