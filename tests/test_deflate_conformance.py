"""DEFLATE conformance on the CPU: the hand-built corpus of deflate_corpus.py (streams zlib never writes) through
zlib and through the inflate kernels' host model (tools/inflate_model.cpp, which compiles the decoder of
ngs_b200/csrc/inflate_lane.cuh for the CPU and restates the resolve kernel's warp algorithm).

Valid cases must decode to their intended bytes at all 16 output alignments; invalid ones must be failed by the decoder
without a byte written outside the block, and rejected by zlib.  What is deliberately not pinned (zlib and the
reference's miniz_oxide disagree) is listed in deflate_corpus.py's docstring."""
import struct
import subprocess
import zlib

import pytest

import deflate_corpus as dc
import deflate_writer as dw
from bamutil import bgzf_block, rec
from test_inflate_model import model  # noqa: F401  (fixture: the compiled host model)

VALID = dc.valid_cases()
INVALID = dc.invalid_cases()


def _raw(blk):
    """(DEFLATE payload, CRC32, ISIZE) of one BGZF block."""
    xlen = struct.unpack_from("<H", blk, 10)[0]
    crc, isize = struct.unpack_from("<II", blk, len(blk) - 8)
    return blk[12 + xlen:-8], crc, isize


# ------------------------------------------------------------------ the writer
def test_canonical_codes_follow_rfc1951_example():
    # RFC 1951 section 3.2.2: lengths (3, 3, 3, 3, 3, 2, 4, 4) for A..H
    assert dw.canonical_codes([3, 3, 3, 3, 3, 2, 4, 4]) == [0b010, 0b011, 0b100, 0b101, 0b110, 0b00, 0b1110, 0b1111]


@pytest.mark.parametrize("max_len", [7, 9, 15])
def test_limited_lengths_are_complete_and_bounded(max_len):
    freqs = [1 << min(i, 40) for i in range(60)] + [0] * 5  # a skew that wants codes far longer than max_len
    lens = dw.limited_lengths(freqs, max_len)
    assert max(lens) == max_len and dw.kraft(lens) == 1 << 15
    assert all((l == 0) == (f == 0) for l, f in zip(lens, freqs))


def test_lz77_round_trip_on_bam_records():
    raw = b"".join(rec(name=f"r{i}", flag=0, ref=0, pos=100 * i, cigar="50M", seq="ACGT" * 12 + "AC", qual=[30] * 50)[0]
                   for i in range(60))
    toks = dw.lz77(raw)
    assert dw.expand(toks) == raw and any(not isinstance(t, int) for t in toks)
    for d in (dw.Deflate().fixed(toks, final=True), dw.Deflate().dynamic(toks, final=True, max_bits=10)):
        assert zlib.decompress(d.getvalue(), -15) == raw


def test_bgzf_wrap_matches_bamutil_framing():
    p = b"ACGT" * 100
    ours = dw.bgzf_wrap(dw.Deflate().stored(p, final=True).getvalue(), p)
    theirs = bgzf_block(p, level=0)
    assert ours[:12] == theirs[:12] and ours[12:16] == theirs[12:16] and ours[-8:] == theirs[-8:]
    assert zlib.decompress(_raw(ours)[0], -15) == p


@pytest.mark.parametrize("name,blocks", VALID, ids=[n for n, _ in VALID])
def test_valid_case_decodes_with_zlib(name, blocks):
    for blk, payload in blocks:
        data, crc, isize = _raw(blk)
        o = zlib.decompressobj(-15)
        assert o.decompress(data) == payload and o.eof and not o.unused_data
        assert isize == len(payload) and crc == zlib.crc32(payload)


@pytest.mark.parametrize("name,blk", INVALID, ids=[n for n, _ in INVALID])
def test_invalid_case_is_rejected_by_zlib(name, blk):
    data, _, isize = _raw(blk)
    o = zlib.decompressobj(-15)
    try:
        out = o.decompress(data)
    except zlib.error:
        return
    assert not (o.eof and len(out) == isize), "zlib decodes the stream to ISIZE bytes"


# ------------------------------------------------------------------ the host model of the kernels
def test_model_decodes_the_valid_corpus_at_every_output_alignment(model, tmp_path):  # noqa: F811
    path = tmp_path / "valid.bgzf"
    n, _ = dc.write_corpus(path, VALID)
    r = subprocess.run([model, str(path), "--all-alignments"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert f"blocks {n}," in r.stdout and "bad 0" in r.stdout


@pytest.mark.parametrize("name,blk", INVALID, ids=[n for n, _ in INVALID])
def test_model_rejects_invalid_case(model, tmp_path, name, blk):  # noqa: F811
    path = tmp_path / f"{name}.bgzf"
    path.write_bytes(blk)
    r = subprocess.run([model, str(path), "--expect-reject"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "reject: 1 blocks, 1 rejected, bad 0" in r.stdout
