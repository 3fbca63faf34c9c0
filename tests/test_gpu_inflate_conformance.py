"""DEFLATE conformance of the GPU inflate (inflate_decode_kernel + inflate_resolve_kernel) on the hand-built corpus of
deflate_corpus.py: streams zlib never writes, decoded by the device build of the decoder (its __byte_perm / __brev /
funnel-shift / __ldg branches) and by the resolve kernel itself rather than its host restatement.

  * every valid case inflates to zlib's bytes, with the cases interleaved so that the 32 lanes of a warp decode
    different shapes (header counts from 1 to 400 per BGZF block);
  * BAM records encoded through the writer's shapes give the oracle's integers, CRC32 on, at launch_blocks 0 and 3;
  * every invalid case fails with NGSQ_E_BAD_BLOCK, both through ngsq_inflate_to_host and in a full run, and the oracle
    (zlib) rejects the file too."""
import numpy as np
import pytest

import deflate_corpus as dc
import deflate_writer as dw
from bamutil import EOF_BLOCK, as_u8, rec, write_bam
from helpers import OracleError, assert_same_ints, engine_ints, oracle_ints

pytestmark = pytest.mark.gpu
REFS = [("chr1", 200000), ("chr2", 50000)]
VALID = dc.valid_cases()
INVALID = dc.invalid_cases()


def _interleaved(cases):
    """BGZF blocks of all cases, round-robin over the cases: neighbouring blocks (lanes of one warp) differ in shape."""
    queues = [list(blocks) for _, blocks in cases]
    out = []
    while any(queues):
        for q in queues:
            if q:
                out.append(q.pop(0))
    return out


@pytest.mark.parametrize("order", ["forward", "reversed"])
def test_valid_corpus_inflates_to_zlib_bytes(order):
    from ngs_b200 import ffi
    blocks = _interleaved(VALID if order == "forward" else VALID[::-1])
    data = as_u8(b"".join(b for b, _ in blocks))
    want = b"".join(p for _, p in blocks)
    got = ffi.Engine().inflate_to_host(data)
    assert got.size == len(want)
    if got.tobytes() != want:
        o = 0
        names = {id(b): n for n, bl in VALID for b, _ in bl}
        for b, p in blocks:
            assert got[o:o + len(p)].tobytes() == p, f"case {names[id(b)]}: bytes differ"
            o += len(p)


# ------------------------------------------------------------------ BAM records through the writer's shapes
def _records(n=700, seed=3):
    rng = np.random.default_rng(seed)
    out = []
    for ref in (0, 1):
        pos = 0
        for i in range(n // 2):
            pos += int(rng.integers(0, 150))
            L = int(rng.integers(30, 200))
            seq = "".join(rng.choice(list("ACGTN"), size=L, p=[0.27, 0.22, 0.22, 0.27, 0.02]))
            out.append(rec(name=f"r{ref}_{i}", flag=int(rng.choice([0x63, 0x93, 0x53, 0xA3, 0x0, 0x10])), ref=ref, pos=pos,
                           mapq=int(rng.choice([0, 20, 60])), cigar=rng.choice([f"{L}M", f"5S{L - 5}M", f"{L - 10}M4I6M"]),
                           next_ref=ref, next_pos=pos + 120, tlen=int(rng.integers(-600, 600)), seq=seq,
                           qual=rng.integers(2, 42, size=L).tolist(), aux=b"NMC\x02" if i % 3 else b""))
    return out


def _skewed_lengths(toks):
    """15-bit-limited literal/length code from exponentially skewed symbol counts: the rarest symbols get 15-bit codes."""
    f = [0] * 286
    for s, _ in dw.Deflate._symbols(toks, True):
        if s[0] == "ll":
            f[s[1]] += 1
    ranked = sorted((s for s in range(286) if f[s]), key=lambda s: -f[s])
    w = [0] * 286
    for r, s in enumerate(ranked):
        w[s] = 1 << max(40 - r, 0)
    return dw.limited_lengths(w, 15)


def _many_blocks(toks, payload):
    """The tokens cut into runs of 40, written as stored / fixed / dynamic blocks in turn, then an empty final stored."""
    d, o = dw.Deflate(), 0
    for k, i in enumerate(range(0, len(toks), 40)):
        run = toks[i:i + 40]
        n = sum(1 if isinstance(t, int) else t[0] for t in run)
        [lambda: d.stored(payload[o:o + n]), lambda: d.fixed(run), lambda: d.dynamic(run, max_bits=9)][k % 3]()
        o += n
    return d.stored(b"", final=True)


SHAPES = {
    "fixed": lambda toks, p: dw.Deflate().fixed(toks, final=True),
    "dynamic": lambda toks, p: dw.Deflate().dynamic(toks, final=True),
    "len15": lambda toks, p: dw.Deflate().dynamic(toks, final=True, ll_lens=_skewed_lengths(toks)),
    "many_blocks": _many_blocks,
    "literal_only_untrimmed": lambda toks, p: dw.Deflate().dynamic(list(p), final=True, d_lens=[0], hlit=286, hdist=30,
                                                                   hclen=19, rle="literal"),
    "stored": lambda toks, p: dw.Deflate().stored(p).stored(b"", final=True),
}


def _writer_blocker(i, payload):
    toks = dw.lz77(payload)
    name = list(SHAPES)[i % len(SHAPES)]
    return dw.bgzf_wrap(SHAPES[name](toks, payload).getvalue(), payload)


@pytest.fixture(scope="module")
def writer_bam():
    bam, bai = write_bam(REFS, _records(), block_payload=[4000, 977, 6000, 2500, 65000, 1, 3333], blocker=_writer_blocker)
    return as_u8(bam), as_u8(bai)


@pytest.mark.parametrize("launch_blocks", [0, 3])
def test_full_run_on_records_encoded_by_the_writer(writer_bam, launch_blocks):
    b, i = writer_bam
    want = oracle_ints(b, i, gc_seed=5)
    got = engine_ints(b, gc_seed=5, crc=True, launch_blocks=launch_blocks)
    assert got["stats"]["records"] == 700
    assert_same_ints(got, want)


# ------------------------------------------------------------------ invalid streams
@pytest.fixture(scope="module")
def valid_prefix():
    """A BAM whose records fill more than 64 KiB of stored blocks, so that the header read (which inflates the first
    64 KiB) never reaches the invalid block appended after them."""
    bam, bai = write_bam(REFS, _records(300, seed=4), level=0, with_eof=False)
    assert len(bam) > 1 << 16
    return bam, bai


@pytest.mark.parametrize("name,blk", INVALID, ids=[n for n, _ in INVALID])
def test_invalid_case_is_a_bad_block(valid_prefix, name, blk):
    from ngs_b200 import ffi
    with pytest.raises(ffi.NgsqError) as ei:
        ffi.Engine().inflate_to_host(as_u8(blk))
    assert ei.value.code == -4, ei.value
    bam, bai = valid_prefix
    b, i = as_u8(bam + blk + EOF_BLOCK), as_u8(bai)
    with pytest.raises(OracleError):
        oracle_ints(b, i)
    with pytest.raises(ffi.NgsqError) as ei:
        engine_ints(b, crc=True)
    assert ei.value.code == -4, ei.value
