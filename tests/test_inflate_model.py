"""CPU check of the inflate kernel's decoder logic: ngs_b200/csrc/inflate_lane.cuh (the per-lane
canonical Huffman decoder the CUDA decode kernel runs, compiled for the host by
tools/inflate_model.cpp) plus the resolve pass — a scalar one at the first output alignment, a lane-by-lane
restatement of the resolve kernel's warp algorithm (32-token batches, dependency masks, rounds, 8-byte copy
steps) at the second — must reproduce zlib's bytes on stored / fixed / dynamic / multi-block DEFLATE streams.  Test tooling only:
nothing under ngs_b200/ links or calls this."""
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

from bamutil import bgzf_block

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def model(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("model") / "inflate_model")
    subprocess.run(["g++", "-O2", "-std=c++17", "-DNGSQ_HOST_MODEL", "-Wno-unknown-pragmas",
                    "-I", os.path.join(ROOT, "ngs_b200", "csrc"), "-o", exe, os.path.join(ROOT, "tools", "inflate_model.cpp"), "-lz"], check=True)
    return exe


def _multi_block_member(pl: bytes) -> bytes:
    """One BGZF member holding several DEFLATE blocks (dynamic, empty stored from the flushes, final)."""
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    third = len(pl) // 3
    data = co.compress(pl[:third]) + co.flush(zlib.Z_FULL_FLUSH)
    data += co.compress(pl[third:2 * third]) + co.flush(zlib.Z_SYNC_FLUSH)
    data += co.compress(pl[2 * third:]) + co.flush()
    return struct.pack("<4BI2BH2BHH", 0x1f, 0x8b, 8, 4, 0, 0, 0xff, 6, 66, 67, 2, len(data) + 25) + data + \
        struct.pack("<II", zlib.crc32(pl), len(pl))


def test_decoder_matches_zlib_on_edge_streams(model, tmp_path):
    rng = np.random.default_rng(5)
    out = b""
    n_blocks = 0
    for i in range(36):
        n = int(rng.choice([1, 2, 3, 17, 100, 1000, 30000, 65280, 65535, 65536]))
        kind = i % 6
        if kind == 0:
            p = bytes(rng.choice(list(b"ACGT"), size=n).astype(np.uint8))
        elif kind == 1:
            p = bytes(rng.integers(0, 256, size=min(n, 60000), dtype=np.uint8))
        elif kind == 2:
            p = b"A" * n
        elif kind == 3:
            p = (b"abc" * (n // 3 + 1))[:n]
        elif kind == 4:
            p = bytes(rng.integers(0, 256, size=min(n, 60000), dtype=np.uint8))
        else:
            p = (bytes(rng.choice(list(b"ACGTN"), size=50).astype(np.uint8)) * (n // 50 + 1))[:n]
        for lvl, strat in [(6, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_DEFAULT_STRATEGY), (0, zlib.Z_DEFAULT_STRATEGY),
                           (6, zlib.Z_FIXED), (9, zlib.Z_HUFFMAN_ONLY), (6, zlib.Z_RLE)]:
            try:
                out += bgzf_block(p, lvl, strat)
                n_blocks += 1
            except AssertionError:  # does not fit one BGZF block at this level
                pass
        if 10 < len(p) < 60000:
            out += _multi_block_member(p)
            n_blocks += 1
    path = tmp_path / "edge.bgzf"
    path.write_bytes(out)
    r = subprocess.run([model, str(path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert f"blocks {n_blocks}," in r.stdout and "bad 0" in r.stdout


def test_decoder_matches_zlib_on_synthetic_bam(model, tmp_path):
    from ngs_b200 import ffi
    for level in (1, 6):
        bam, _, info = ffi.synth_bam(1, 20000, level=level)
        path = tmp_path / f"s{level}.bam"
        path.write_bytes(bam.tobytes())
        r = subprocess.run([model, str(path)], capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        assert "bad 0" in r.stdout


def test_decoder_survives_corrupted_streams(model, tmp_path):
    """Bit flips in the DEFLATE payload: the decoder must reject the block or finish it, never write
    outside the block's output range, never mark matches beyond it, never emit an unresolvable token
    (the resolve kernel trusts tokens of blocks that decoded without error) and never run away."""
    from ngs_b200 import ffi
    bam, _, _ = ffi.synth_bam(1, 6000, level=6)
    out = bam.tobytes()
    for payload, lvl, strat in [(b"ACGT" * 9000, 6, zlib.Z_FIXED), (bytes(range(256)) * 200, 0, zlib.Z_DEFAULT_STRATEGY),
                                (b"A" * 65000, 9, zlib.Z_DEFAULT_STRATEGY)]:
        out += bgzf_block(payload, lvl, strat)
    path = tmp_path / "fuzz.bgzf"
    path.write_bytes(out)
    r = subprocess.run([model, str(path), "--fuzz", "60"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "bad 0" in r.stdout
