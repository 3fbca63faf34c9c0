"""Cuts of a BAM without an index on CPU (ngs_b200/host/bam.hpp: next_block_start, plan_shards_unindexed), through
tests/cpp/host_unindexed.cpp with a record finder backed by the truth: block starts are found by their signature and a chain
of blocks behind it, a signature inside a block's payload is skipped, and the plan is the one its rule gives (targets
snapped to the next block start, moved to the first record from there, repeated anchors and targets without a record left
out) with the split set of every contig that has records on both sides of a cut."""
import bisect
import os
import struct
import subprocess
import zlib

import pytest

import bamutil

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("unindexed") / "host_unindexed")
    subprocess.run(["g++", "-O1", "-std=c++17", "-o", out, os.path.join(ROOT, "tests", "cpp", "host_unindexed.cpp"),
                    "-L" + os.path.join(ROOT, "ngs_b200"), "-lngs_cuda", "-Wl,-rpath," + os.path.join(ROOT, "ngs_b200")], check=True)
    return out


def walk(raw: bytes):
    """(block starts, first record voffset, [(voffset, refID)] of every record), inflating with zlib."""
    from ngs_b200 import formats
    coffs, ustarts, data, off = [], [], bytearray(), 0
    while off < len(raw):
        bsize = int.from_bytes(raw[off + 16:off + 18], "little") + 1
        coffs.append(off)
        ustarts.append(len(data))
        data += zlib.decompress(raw[off + 18:off + bsize - 8], -15)
        off += bsize

    def voff(u):
        k = bisect.bisect_right(ustarts, u) - 1
        while k + 1 < len(ustarts) and ustarts[k + 1] == u:  # an offset at a block's end names the next non-empty block
            k += 1
        return (coffs[k] << 16) | (u - ustarts[k])

    _, _, hlen = formats.parse_bam_header(bytes(data))
    recs, o = [], hlen
    while o + 4 <= len(data):
        n = struct.unpack_from("<i", data, o)[0]
        recs.append((voff(o), struct.unpack_from("<i", data, o + 4)[0]))
        o += 4 + n
    return coffs, voff(hlen), recs


def _files():
    from ngs_b200 import ffi
    out = {}
    for shape in range(4):
        out[f"shape{shape}"] = bytes(ffi.synth_bam(shape, 2500 if shape == 2 else 40000, level=1)[0])
    return out


FILES = None


def _file(name):
    global FILES
    if FILES is None:
        FILES = _files()
    return FILES[name]


@pytest.mark.parametrize("name", ["shape0", "shape1", "shape2", "shape3"])
def test_block_starts_of_bamgen_files(exe, tmp_path, name):
    raw = _file(name)
    p = tmp_path / "x.bam"
    p.write_bytes(raw)
    got = [int(x) for x in subprocess.run([exe, "blocks", str(p)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == walk(raw)[0]


def test_a_signature_that_does_not_chain_is_skipped(exe, tmp_path):
    """Stored blocks (level 0) keep a record's bytes as they are: a read whose auxiliary data holds a BGZF header puts the
    signature in the file, inside a block's payload.  Its BSIZE points at bytes that are no block header."""
    fake = bytes.fromhex("1f8b08040000000000ff0600424302003f00") + b"\x07" * 64
    recs = [bamutil.rec(name=f"r{i}", flag=0, ref=0, pos=100 + i, mapq=30, cigar="10M", seq="ACGTACGTAC", qual=[30] * 10,
                        aux=b"XBZ" + fake + b"\x00" if i == 3 else b"") for i in range(8)]
    raw, _ = bamutil.write_bam([("chr1", 10000)], recs, level=0)
    at = raw.find(fake)
    assert at > 0
    blocks = walk(raw)[0]
    assert at not in blocks
    p = tmp_path / "d.bam"
    p.write_bytes(raw)
    got = [int(x) for x in subprocess.run([exe, "blocks", str(p)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == blocks


def _expected(raw, first, recs, n):
    """The plan's cuts by its rule, from the truth."""
    blocks = walk(raw)[0]
    base = first >> 16
    cuts, dropped = [], 0
    for k in range(1, n):
        target = base + (len(raw) - base) * k // n
        j = bisect.bisect_left(blocks, target)
        anchor = None
        if j < len(blocks):
            i = bisect.bisect_left(recs, (blocks[j] << 16, -(1 << 31)))
            anchor = recs[i] if i < len(recs) else None
        if anchor is None or anchor[0] <= (cuts[-1][0] if cuts else first):
            dropped += 1
        else:
            cuts.append(anchor)
    return cuts, dropped


@pytest.mark.parametrize("n", [2, 3, 5, 8, 40, 0])  # 0: twice as many shards as blocks
@pytest.mark.parametrize("name", ["shape0", "shape1", "shape2", "shape3"])
def test_the_plan_with_a_truth_backed_finder(exe, tmp_path, name, n):
    raw = _file(name)
    blocks, first, recs = walk(raw)
    many = n == 0
    n = n or 2 * len(blocks)
    p, t = tmp_path / "x.bam", tmp_path / "truth.txt"
    p.write_bytes(raw)
    t.write_text("".join(f"{v} {r}\n" for v, r in recs))
    out = subprocess.run([exe, "plan", str(p), str(first), str(n), str(t)], capture_output=True, text=True, check=True).stdout
    assert not out.startswith("error"), out
    lines = out.splitlines()
    rows = [[int(x) for x in ln.split()] for ln in lines[:n]]
    split = [int(x) for x in lines[n].split()[1:]]
    dropped = int(lines[n + 1].split()[1])
    cuts, want_dropped = _expected(raw, first, recs, n)
    live = [r for r in rows if not r[2]]
    assert [r[0] for r in live] == [first] + [v for v, _ in cuts]        # the rule's anchors, strictly increasing
    assert all(a[1] == b[0] for a, b in zip(live, live[1:])) and live[-1][1] == 0
    assert len(rows) == n and all(r[2] for r in rows[len(live):])      # left-out cuts become empty shards at the end
    assert dropped == want_dropped == n - len(live)
    starts = {v for v, _ in recs}
    assert all(r[0] in starts for r in live[1:])
    assert split == sorted({r for _, r in cuts if r >= 0})
    # complete: every contig with records on both sides of a cut is declared
    for v, _ in cuts:
        before = {r for w, r in recs if w < v and r >= 0}
        after = {r for w, r in recs if w >= v and r >= 0}
        assert before & after <= set(split)
    if many:
        assert dropped > len(blocks)  # more targets than blocks: anchors repeat
