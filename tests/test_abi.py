"""The C-ABI library loads and exports every symbol include/ngs_cuda.h declares; host-side
entry points (K1 BGZF framing) work without a GPU; without a device the engine fails loudly."""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from bamutil import EOF_BLOCK, as_u8, bgzf_block, rec, write_bam

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_and_library_agree():
    from ngs_b200 import ffi
    lib = ffi.load_library()
    hdr = open(os.path.join(ROOT, "include", "ngs_cuda.h")).read()
    declared = set(re.findall(r"\b(ngsq_[a-z0-9_]+)\s*\(", hdr))
    declared -= {"ngsq_engine", "ngsq_config", "ngsq_block", "ngsq_stats", "ngsq_cov_ints"}
    assert declared, "no declarations found"
    for name in sorted(declared):
        assert hasattr(lib, name), f"{name} declared in include/ngs_cuda.h but not exported"
    assert declared == set(ffi.EXPORTED)  # nothing bound that the header does not declare, and vice versa
    assert lib.ngsq_version() == 0x000100


def test_struct_layouts_match_header():
    from ngs_b200 import ffi
    assert C.sizeof(ffi.Block) == 24
    assert C.sizeof(ffi.Config) == 64
    assert C.sizeof(ffi.CovInts) == 16 + 2049 * 8
    assert C.sizeof(ffi.Stats) == 96  # 5 u64, 6 floats, 2 u32, 5 floats (decode / resolve / reduce / edits / tail), 1 u32


def test_create_fails_loudly_without_gpu():
    """In a child process that sees no device (CUDA_VISIBLE_DEVICES=""), so the check also runs where a GPU is present."""
    child = ("import sys\n"
             f"sys.path.insert(0, {ROOT!r})\n"
             "from ngs_b200 import ffi\n"
             "try:\n"
             "    ffi.Engine()\n"
             "except ffi.NgsqError as ex:\n"
             "    print(ex.code, ex)\n")
    r = subprocess.run([sys.executable, "-c", child], env={**os.environ, "CUDA_VISIBLE_DEVICES": ""}, capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stderr
    code, _, message = r.stdout.strip().partition(" ")
    assert code == "-2" and "no CPU fallback" in message, r.stdout


def test_bgzf_walk_on_host():
    from ngs_b200 import ffi
    payloads = [b"a" * 1000, b"", os.urandom(65536 - 100), b"xyz"]
    raw = b"".join(bgzf_block(p, extra_subfield=(i == 1)) for i, p in enumerate(payloads)) + EOF_BLOCK
    data = as_u8(raw)
    blocks, n, used = ffi.bgzf_walk(data, file_off=1 << 20)
    assert n == 5 and used == len(raw)
    assert [blocks[i].isize for i in range(n)] == [1000, 0, 65436, 3, 0]
    assert blocks[0].coffset == 1 << 20 and blocks[1].hdr_len == 25 and blocks[0].hdr_len == 18
    assert sum(blocks[i].csize for i in range(n)) == len(raw)
    import zlib
    assert blocks[2].crc32 == zlib.crc32(payloads[2]) & 0xFFFFFFFF
    # a trailing partial block is reported through `consumed`, not as an error
    _, n2, used2 = ffi.bgzf_walk(data[:-5])
    assert n2 == 4 and used2 == len(raw) - 28


def test_bgzf_walk_rejects_bad_magic():
    from ngs_b200 import ffi
    raw = bytearray(bgzf_block(b"hello") + EOF_BLOCK)
    raw[1] = 0x00
    with pytest.raises(ffi.NgsqError):
        ffi.bgzf_walk(as_u8(bytes(raw)))


def test_synthetic_writer_is_deterministic_and_valid():
    import gzip
    from ngs_b200 import ffi, formats
    a, ai, info = ffi.synth_bam(0, 5000, level=6, threads=1)
    b, bi, _ = ffi.synth_bam(0, 5000, level=6, threads=4)
    assert np.array_equal(a, b) and np.array_equal(ai, bi), "output must not depend on the thread count"
    plain = gzip.decompress(a.tobytes())
    assert len(plain) == info["inflated_bytes"]
    text, refs, hlen = formats.parse_bam_header(plain)
    assert [r[0] for r in refs] == ["chr1", "chr2", "chrM"] and hlen == info["header_bytes"]
    assert "@SQ\tSN:chr1\tLN:20000000" in text
    bai = formats.parse_bai(ai.tobytes())
    assert len(bai.refs) == 3 and bai.n_no_coor == 50
    assert sum(r.n_mapped + r.n_unmapped for r in bai.refs) + bai.n_no_coor == 5000

