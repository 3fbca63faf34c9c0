"""The records of a coordinate-sorted BAM written again in another order (for `qc --cuda-any-order`): at random, by read name
(the order of a queryname sort or a collate), or reversed.  The header is kept byte for byte; the records are packed into
BGZF blocks of `block_payload` bytes, so they straddle block boundaries wherever the sizes fall."""
import struct
import zlib

import numpy as np

from bamutil import EOF_BLOCK, bgzf_block

ORDERS = ("random", "queryname", "reversed")


def split_records(bam: bytes):
    """(header bytes, [record bytes]) of a BAM, inflated with zlib."""
    from ngs_b200 import formats
    raw, data, off = bytes(bam), bytearray(), 0
    while off < len(raw):
        bsize = int.from_bytes(raw[off + 16:off + 18], "little") + 1
        data += zlib.decompress(raw[off + 18:off + bsize - 8], -15)
        off += bsize
    _, _, hlen = formats.parse_bam_header(bytes(data))
    recs, o = [], hlen
    while o + 4 <= len(data):
        n = struct.unpack_from("<i", data, o)[0]
        recs.append(bytes(data[o:o + 4 + n]))
        o += 4 + n
    assert o == len(data)
    return bytes(data[:hlen]), recs


def _name(r: bytes) -> bytes:
    return r[36:36 + r[12] - 1]


def order_of(recs, kind, seed=0):
    """Indices of recs in the new order."""
    n = len(recs)
    if kind == "random":
        return list(np.random.default_rng(seed).permutation(n))
    if kind == "queryname":  # mates next to each other, read 1 before read 2; ties keep the file order
        return sorted(range(n), key=lambda i: (_name(recs[i]), struct.unpack_from("<H", recs[i], 18)[0] & 0xC0, i))
    if kind == "reversed":
        return list(range(n))[::-1]
    raise ValueError(kind)


def reorder(bam, kind, seed=0, block_payload=0xFF00, level=6):
    """U: the header and records of bam, the records in order `kind`; returns (u8 array, the order)."""
    hdr, recs = split_records(bam)
    order = order_of(recs, kind, seed)
    stream = b"".join(recs[i] for i in order)
    out = bytearray(bgzf_block(hdr, level))
    for o in range(0, len(stream), block_payload):
        out += bgzf_block(stream[o:o + block_payload], level)
    out += EOF_BLOCK
    return np.frombuffer(bytes(out), dtype=np.uint8).copy(), order
