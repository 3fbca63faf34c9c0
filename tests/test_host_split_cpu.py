"""The C++ host driver's intra-contig shard planner (ngs_b200/host/bam.hpp: plan_shards_split, choose_shards) on CPU, and its
Python mirror (ngs_b200/formats.py).  For any number of devices the shards must be a contiguous partition of the records,
from the first one to EOF, cut at record starts taken from the BAI; the split set must be exactly the contigs with records on
both sides of a cut (found here by walking the records themselves); byte ranges must hold whole BGZF blocks; no shard may be
empty while anchors remain."""
import bisect
import os
import struct
import subprocess
import zlib

import numpy as np
import pytest

import bamutil

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_SHARDS = [1, 2, 3, 4, 8, 24, 40]


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("split") / "host_split")
    subprocess.run(["g++", "-O1", "-std=c++17", "-o", out, os.path.join(ROOT, "tests", "cpp", "host_split.cpp"),
                    "-L" + os.path.join(ROOT, "ngs_b200"), "-lngs_cuda", "-Wl,-rpath," + os.path.join(ROOT, "ngs_b200")], check=True)
    return out


def walk(raw: bytes):
    """(first record voffset, [(voffset, refID)] of every record, block start offsets) by inflating the file with zlib."""
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

    _, refs, hlen = formats.parse_bam_header(bytes(data))
    walk.refs = refs  # the header's (name, length) list of the last file walked
    recs, o = [], hlen
    while o + 4 <= len(data):
        n = struct.unpack_from("<i", data, o)[0]
        recs.append((voff(o), struct.unpack_from("<i", data, o + 4)[0]))
        o += 4 + n
    return voff(hlen), recs, coffs


def single_contig_bam():
    """One 2 Mb contig: short reads every few hundred bases, a deep pile and some long reads."""
    rng = np.random.default_rng(7)
    L = 2_000_000
    pos = np.sort(np.concatenate([rng.integers(0, L - 200, 6000), np.full(300, 700_000)]))
    records = []
    for i, p in enumerate(pos):
        cig = "5000M" if i % 500 == 0 and p < L - 6000 else "100M"
        n = 5000 if cig == "5000M" else 100
        records.append(bamutil.rec(name=f"r{i}", flag=0, ref=0, pos=int(p), mapq=60, cigar=cig, seq="A" * n, qual=[30] * n))
    records.append(bamutil.rec(name="u", flag=4, seq="ACGT", qual=[30] * 4))  # unplaced tail
    return bamutil.write_bam([("chr1", L)], records, level=1)


@pytest.fixture(scope="module", params=["shape0", "shape1", "shape2", "shape3", "single"])
def case(request, tmp_path_factory):
    from ngs_b200 import ffi, formats
    d = tmp_path_factory.mktemp("splitcase")
    if request.param == "single":
        bam, bai = single_contig_bam()
        n_ref = 1
    else:
        shape = int(request.param[-1])
        b, i, info = ffi.synth_bam(shape, 3000 if shape == 2 else 60000, level=1)
        bam, bai, n_ref = b.tobytes(), i.tobytes(), info["n_ref"]
    (d / "x.bam").write_bytes(bam)
    (d / "x.bam.bai").write_bytes(bai)
    first, recs, coffs = walk(bam)
    LENGTHS[str(d / "x.bam")] = ",".join(str(l) for _, l in walk.refs)
    return request.param, str(d / "x.bam"), first, n_ref, formats.parse_bai(bai), bam, recs, coffs


LENGTHS = {}  # BAM path -> its reference lengths as host_split takes them


def run(exe, path, first, n_ref, n):
    out = subprocess.run([exe, path, str(first), str(n_ref), str(n), LENGTHS.get(path, "")], capture_output=True, text=True,
                         check=True).stdout
    assert not out.startswith("error"), out
    lines = out.splitlines()
    rows = [[int(x) for x in ln.split()] for ln in lines[:-3]]
    split = [int(x) for x in lines[-3].split()[1:]]
    anchors = [int(x) for x in lines[-2].split()[1:]]
    pick = lines[-1].split()
    return rows, split, anchors, pick[1], [int(x) for x in pick[2:]]


@pytest.mark.parametrize("n_shards", N_SHARDS)
def test_split_plan_partitions_the_records(exe, case, n_shards):
    from ngs_b200 import formats
    name, path, first, n_ref, bai, raw, recs, coffs = case
    rows, split, anchors, _, _ = run(exe, path, first, n_ref, n_shards)
    assert len(rows) == n_shards
    assert anchors == formats.bai_anchors(bai)
    live = [r for r in rows if not r[2]]
    assert live[0][0] == first == recs[0][0] and live[-1][1] == 0                  # first record .. EOF
    starts = {v for v, _ in recs}
    cuts = [a[1] for a in live[:-1]]
    for a, b in zip(live, live[1:]):
        assert a[1] == b[0] and a[1] > a[0]                                         # contiguous, strictly increasing
        assert a[1] in anchors and a[1] in starts                                   # cut at a BAI anchor = a record start
    blocks = set(coffs)
    for r in live:                                                                  # whole BGZF blocks through the end record
        assert r[3] in blocks and (r[4] == len(raw) or r[4] in blocks) and r[3] < r[4]
        assert r[3] == r[0] >> 16 and (r[1] == 0 or r[4] > r[1] >> 16 or (r[1] & 0xFFFF) == 0)
    n_cand = sum(1 for v in anchors if v > first)
    assert len(live) == min(n_shards, 1 + n_cand)                                   # nobody idle while anchors remain
    # the split set, from the records: contigs with records on both sides of some cut
    want = set()
    for v in cuts:
        before = {ref for o, ref in recs if o < v and ref >= 0}
        after = {ref for o, ref in recs if o >= v and ref >= 0}
        want |= before & after
    assert split == sorted(want)
    # every shard lists the references it holds records of
    bounds = [r[0] for r in live] + [1 << 64]
    for i, r in enumerate(live):
        held = sorted({ref for o, ref in recs if bounds[i] <= o < bounds[i + 1] and ref >= 0})
        assert r[5:] == held, (i, r[5:], held)
    # the Python mirror agrees
    hdr = formats.BamHeader("", [("", 0)] * n_ref, 0, first)
    shards, py_split = formats.plan_shards_split(hdr, bai, n_shards, len(raw))
    assert py_split == split
    assert [(s.first_voffset, s.end_voffset, s.contigs) for s in shards] == [(r[0], r[1], r[5:]) for r in rows]


# choose_shards keeps the contig-aligned plan while it is balanced and leaves no device idle
CHOICES = {"shape0": [(1, "contig"), (4, "split")], "shape1": [(1, "contig"), (2, "contig")], "shape2": [(1, "contig")],
           "shape3": [(1, "contig")], "single": [(1, "contig"), (2, "split"), (4, "split")]}


def test_choose_shards(exe, case):
    name, path, first, n_ref, bai, raw, recs, coffs = case
    for n, want in CHOICES[name]:
        rows, split, _, pick, pick_split = run(exe, path, first, n_ref, n)
        assert pick == want, (name, n)
        assert pick_split == (split if want == "split" else []), (name, n)


def test_choose_keeps_whole_contigs_when_the_merge_outweighs_the_balance(exe, tmp_path):
    """The 25-contig WGS shape at 8 devices: its largest contig-aligned shard is 26 % above the mean, but cutting inside
    contigs would split 7 contigs whose difference arrays outweigh twice a balanced shard's compressed bytes, so the
    contig-aligned plan stays.  At 2 devices the single-contig file always takes the split plan (one device would idle)."""
    from ngs_b200 import ffi
    b, i, info = ffi.synth_bam(1, 2_000_000, level=1, threads=8)
    raw = b.tobytes()
    (tmp_path / "w.bam").write_bytes(raw)
    (tmp_path / "w.bam.bai").write_bytes(i.tobytes())
    first, _, _ = walk(raw)
    path = str(tmp_path / "w.bam")
    LENGTHS[path] = ",".join(str(l) for _, l in walk.refs)
    _, split, _, pick, pick_split = run(exe, path, first, info["n_ref"], 8)
    assert len(split) == 7                      # what the split plan would cut
    assert pick == "contig" and pick_split == []
    LENGTHS[path] = ""  # reference lengths unknown: the merge looks free
    _, split, _, pick, _ = run(exe, path, first, info["n_ref"], 8)
    assert pick == "split"                      # without the merge's cost the 26 % imbalance alone would cut inside contigs
