"""The C++ host driver's CSI reader (ngs_b200/host/bam.hpp: parse_csi) on CPU, through tests/cpp/host_csi.cpp: a CSI payload must
give the shard planner what the BAI of the same file gives it.  Per reference the extent and the mapped and unmapped counts
equal the BAI pseudo-bin's, so the contig-aligned plan is the BAI's; every anchor is the start of a record of its reference (at
min_shift 14 a subset of the BAI's anchors), and the plan cut inside contigs partitions the records with the split set the
records give.  htslib-shaped payloads (aux bytes, leaf bins folded into their parents, forward-filled, all-ones and leading zero
loffsets) plan from record starts too, and malformed payloads are refused with a message that names the file."""
import os
import struct
import subprocess

import pytest

import bamutil  # noqa: F401  (tests/ on the path for the helpers below)
from baiutil import micro_bams, oracle_bai
from csiutil import oracle_csi
from test_host_split_cpu import walk

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHIFTS = [12, 14, 16]
N_SHARDS = [2, 3, 5, 8]


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("csi") / "host_csi")
    subprocess.run(["g++", "-O1", "-std=c++17", "-o", out, os.path.join(ROOT, "tests", "cpp", "host_csi.cpp"),
                    "-L" + os.path.join(ROOT, "ngs_b200"), "-lngs_cuda", "-Wl,-rpath," + os.path.join(ROOT, "ngs_b200")], check=True)
    return out


MICRO = ["block_starts", "spanning", "zero_span_unmapped", "bin0", "empty_middle", "unplaced_tail", "header_only", "overhang"]


@pytest.fixture(scope="module", params=["shape0", "shape1", "shape2", "shape3"] + MICRO)
def case(request, tmp_path_factory):
    """(name, BAM path, .bai path, first record voffset, n_ref, [(voffset, refID)] of every record, BAM bytes)"""
    from ngs_b200 import ffi
    d = tmp_path_factory.mktemp("csicase")
    if request.param.startswith("shape"):
        shape = int(request.param[-1])
        bam = ffi.synth_bam(shape, 3000 if shape == 2 else 60000, level=1)[0].tobytes()
    else:
        bam = micro_bams()[request.param][0]
    (d / "x.bam").write_bytes(bam)
    (d / "x.bam.bai").write_bytes(oracle_bai(bam))
    first, recs, _ = walk(bam)
    return request.param, str(d / "x.bam"), str(d / "x.bam.bai"), first, len(walk.refs), recs, bam


def run(exe, bam, index, kind, first, n_ref, n_shards):
    out = subprocess.run([exe, bam, index, kind, str(first), str(n_ref), str(n_shards)], capture_output=True, text=True,
                         check=True).stdout
    if out.startswith("error: "):
        return out[len("error: "):].strip()
    res = {"ref": [], "contig": [], "shard": []}
    for ln in out.splitlines():
        tag, *vals = ln.split()
        vals = [int(x) for x in vals]
        if tag in res:
            res[tag].append(vals)
        else:
            res[tag] = vals
    return res


def csi_file(tmp_path, payload, name="x.csi"):
    p = tmp_path / name
    p.write_bytes(payload)
    return str(p)


# ---------------------------------------------------------------- CSIv1 payloads taken apart and put back together
def split_csi(buf):
    """(min_shift, depth, aux, [[(bin, loffset, [(beg, end)])] per reference in file order], tail bytes)"""
    min_shift, depth, l_aux = struct.unpack_from("<iii", buf, 4)
    aux = buf[16:16 + l_aux]
    o = 16 + l_aux
    n_ref = struct.unpack_from("<i", buf, o)[0]
    o += 4
    refs = []
    for _ in range(n_ref):
        n_bin = struct.unpack_from("<i", buf, o)[0]
        o += 4
        bins = []
        for _ in range(n_bin):
            b, loff, n_chunk = struct.unpack_from("<IQi", buf, o)
            o += 16
            bins.append((b, loff, [struct.unpack_from("<QQ", buf, o + 16 * k) for k in range(n_chunk)]))
            o += 16 * n_chunk
        refs.append(bins)
    return min_shift, depth, aux, refs, buf[o:]


def join_csi(min_shift, depth, aux, refs, tail):
    out = bytearray(b"CSI\x01" + struct.pack("<iii", min_shift, depth, len(aux)) + aux + struct.pack("<i", len(refs)))
    for bins in refs:
        out += struct.pack("<i", len(bins))
        for b, loff, chunks in bins:
            out += struct.pack("<IQi", b, loff, len(chunks))
            for beg, end in chunks:
                out += struct.pack("<QQ", beg, end)
    return bytes(out + tail)


def meta_bin(depth):
    return ((1 << 3 * (depth + 1)) - 1) // 7 + 1


def level_of(b):
    lv = 0
    while b:
        b = (b - 1) >> 3
        lv += 1
    return lv


def bin_bot(b, depth):
    lv = level_of(b)
    return (b - ((1 << 3 * lv) - 1) // 7) << 3 * (depth - lv)


def with_aux(buf):
    """tabix-style meta in the aux field (htslib writes it for indexed text files)"""
    ms, d, _, refs, tail = split_csi(buf)
    names = b"chr1\0chr2\0"
    aux = struct.pack("<iiiiiii", 0, 1, 2, 3, ord("#"), 0, len(names)) + names
    return join_csi(ms, d, aux, refs, tail)


def fold_leaves(buf):
    """htslib's compress_binning: leaf bins folded into their parent, chunks moved, the parent's loffset the minimum"""
    ms, d, aux, refs, tail = split_csi(buf)
    out = []
    first_leaf = ((1 << 3 * d) - 1) // 7
    for bins in refs:
        merged = {}
        for b, loff, chunks in bins:
            key = (b - 1) >> 3 if first_leaf <= b < meta_bin(d) else b
            if key in merged:
                l0, c0 = merged[key]
                merged[key] = (min(l0, loff), sorted(c0 + chunks))
            else:
                merged[key] = (loff, list(chunks))
        out.append([(b, loff, chunks) for b, (loff, chunks) in merged.items()])
    return join_csi(ms, d, aux, out, tail)


def forward_fill(buf):
    """every other bin, in the order of their first windows, takes the loffset of the bin on its left (an empty first window
    filled from the left), and the last one all ones (htslib's unset offset)"""
    ms, d, aux, refs, tail = split_csi(buf)
    out = []
    for bins in refs:
        order = sorted((i for i, (b, _, _) in enumerate(bins) if b != meta_bin(d)), key=lambda i: (bin_bot(bins[i][0], d), bins[i][0]))
        new = list(bins)
        for j in range(1, len(order), 2):
            b, _, chunks = new[order[j]]
            new[order[j]] = (b, new[order[j - 1]][1], chunks)
        if order:
            b, _, chunks = new[order[-1]]
            new[order[-1]] = (b, (1 << 64) - 1, chunks)
        out.append(new)
    return join_csi(ms, d, aux, out, tail)


def leading_zeros(buf):
    """loffset 0 on the first bins of every reference, in the order of their first windows"""
    ms, d, aux, refs, tail = split_csi(buf)
    out = []
    for bins in refs:
        order = sorted((i for i, (b, _, _) in enumerate(bins) if b != meta_bin(d)), key=lambda i: (bin_bot(bins[i][0], d), bins[i][0]))
        new = list(bins)
        for i in order[:max(1, len(order) // 3)]:
            b, _, chunks = new[i]
            new[i] = (b, 0, chunks)
        out.append(new)
    return join_csi(ms, d, aux, out, tail)


HTSLIB_SHAPES = {"aux": with_aux, "folded": fold_leaves, "forward_filled": forward_fill, "leading_zeros": leading_zeros,
                 "all": lambda b: leading_zeros(forward_fill(fold_leaves(with_aux(b))))}


# ---------------------------------------------------------------- checks
def check_anchors(res, recs, csi_payload=None):
    """every anchor starts a record; per reference every loffset the planner keeps starts a record of that reference"""
    ref_of = {v: r for v, r in recs}
    for v in res["anchors"]:
        assert v in ref_of, v
    if csi_payload is not None:
        ms, d, _, refs, _ = split_csi(csi_payload)
        for c, bins in enumerate(refs):
            has, beg, end = res["ref"][c][:3]
            for b, loff, _ in bins:
                if has and b != meta_bin(d) and loff and beg <= loff < end:
                    assert ref_of.get(loff) == c, (c, b, loff)


def check_split_plan(res, recs, first, n_shards):
    rows = res["shard"]
    assert len(rows) == n_shards
    live = [r for r in rows if not r[2]]
    assert live[0][0] == first and live[-1][1] == 0
    starts = {v for v, _ in recs}
    for a, b in zip(live, live[1:]):
        assert a[1] == b[0] and a[1] > a[0]
        assert a[1] in res["anchors"] and a[1] in starts
    n_cand = sum(1 for v in res["anchors"] if v > first)
    assert len(live) == min(n_shards, 1 + n_cand)
    want = set()
    for v in [r[1] for r in live[:-1]]:
        before = {ref for o, ref in recs if o < v and ref >= 0}
        after = {ref for o, ref in recs if o >= v and ref >= 0}
        want |= before & after
    assert res["split"] == sorted(want)
    # the records partition: each one in exactly the shard whose range holds it
    bounds = [r[0] for r in live] + [1 << 64]
    assert sum(sum(1 for o, _ in recs if bounds[i] <= o < bounds[i + 1]) for i in range(len(live))) == len(recs)


# ---------------------------------------------------------------- tests
@pytest.mark.parametrize("min_shift", SHIFTS)
def test_extents_and_contig_plan_equal_the_bai(exe, case, tmp_path, min_shift):
    name, bam, bai, first, n_ref, recs, raw = case
    payload = oracle_csi(raw, min_shift, 0)
    csi = csi_file(tmp_path, payload)
    for n in [1] + N_SHARDS:
        from_csi = run(exe, bam, csi, "csi", first, n_ref, n)
        from_bai = run(exe, bam, bai, "bai", first, n_ref, n)
        assert isinstance(from_csi, dict), from_csi
        assert from_csi["ref"] == from_bai["ref"]
        assert from_csi["contig"] == from_bai["contig"], n


@pytest.mark.parametrize("min_shift", SHIFTS)
def test_anchors_are_record_starts_of_their_reference(exe, case, tmp_path, min_shift):
    name, bam, bai, first, n_ref, recs, raw = case
    payload = oracle_csi(raw, min_shift, 0)
    res = run(exe, bam, csi_file(tmp_path, payload), "csi", first, n_ref, 2)
    check_anchors(res, recs, payload)
    if min_shift == 14:  # each loffset is a linear-index value of the same file
        assert set(res["anchors"]) <= set(run(exe, bam, bai, "bai", first, n_ref, 2)["anchors"])


@pytest.mark.parametrize("min_shift", SHIFTS)
@pytest.mark.parametrize("n_shards", N_SHARDS)
def test_split_plan_partitions_the_records(exe, case, tmp_path, n_shards, min_shift):
    name, bam, bai, first, n_ref, recs, raw = case
    if not recs:
        return
    res = run(exe, bam, csi_file(tmp_path, oracle_csi(raw, min_shift, 0)), "csi", first, n_ref, n_shards)
    check_split_plan(res, recs, first, n_shards)


@pytest.mark.parametrize("shape", sorted(HTSLIB_SHAPES))
def test_htslib_shaped_payloads(exe, case, tmp_path, shape):
    name, bam, bai, first, n_ref, recs, raw = case
    plain = oracle_csi(raw, 14, 0)
    payload = HTSLIB_SHAPES[shape](plain)
    want =run(exe, bam, csi_file(tmp_path, plain, "plain.csi"), "csi", first, n_ref, 3)
    got = run(exe, bam, csi_file(tmp_path, payload), "csi", first, n_ref, 3)
    assert isinstance(got, dict), got
    assert got["ref"] == want["ref"]
    assert got["contig"] == want["contig"]
    check_anchors(got, recs, payload)
    assert set(got["anchors"]) <= set(want["anchors"])
    if recs:
        for n in N_SHARDS:
            check_split_plan(run(exe, bam, csi_file(tmp_path, payload), "csi", first, n_ref, n), recs, first, n)


def test_folding_and_filling_change_the_payload():
    """the rewrites above really produce the shapes they name (on a file with many bins)"""
    from ngs_b200 import ffi
    raw = ffi.synth_bam(0, 20000, level=1)[0].tobytes()
    plain = oracle_csi(raw, 14, 0)
    _, d, _, refs, _ = split_csi(plain)
    folded = split_csi(fold_leaves(plain))[3]
    assert sum(map(len, folded)) < sum(map(len, refs))
    assert any(level_of(b) == d for bins in refs for b, _, _ in bins)
    assert not any(level_of(b) == d for bins in folded for b, _, _ in bins if b != meta_bin(d))
    filled = split_csi(forward_fill(plain))[3]
    assert any((1 << 64) - 1 == loff for bins in filled for _, loff, _ in bins)
    zeros = split_csi(leading_zeros(plain))[3]
    assert sum(loff == 0 for bins in zeros for _, loff, _ in bins) > sum(loff == 0 for bins in refs for _, loff, _ in bins)
    assert split_csi(with_aux(plain))[2]


# ---------------------------------------------------------------- malformed payloads
@pytest.fixture(scope="module")
def small(tmp_path_factory):
    d = tmp_path_factory.mktemp("csibad")
    raw = micro_bams()["empty_middle"][0]
    (d / "x.bam").write_bytes(raw)
    first, recs, _ = walk(raw)
    return str(d / "x.bam"), first, len(walk.refs), oracle_csi(raw, 14, 0)


def refused(exe, small, tmp_path, payload, match, n_ref=None):
    """the payload is refused with a message that names the file and holds one of `match` ('|'-separated)"""
    bam, first, n, _ = small
    path = csi_file(tmp_path, payload, "bad.csi")
    msg = run(exe, bam, path, "csi", first, n if n_ref is None else n_ref, 2)
    assert isinstance(msg, str), f"accepted: {payload[:32]!r}"
    assert path in msg and any(m in msg for m in match.split("|")), msg
    return msg


def test_bad_magic(exe, small, tmp_path):
    good = small[3]
    refused(exe, small, tmp_path, b"BAI\x01" + good[4:], "bad magic")
    refused(exe, small, tmp_path, b"CSI\x02" + good[4:], "bad magic")


def test_truncation_at_every_field(exe, small, tmp_path):
    """every cut in front of the optional n_no_coor is refused (inside a bin's chunks its n_chunk runs past the end); from
    there on the payload is whole"""
    good = small[3]
    for n in range(len(good) - 8):
        refused(exe, small, tmp_path, good[:n], "truncated|n_chunk")
    for n in range(len(good) - 8, len(good) + 1):
        assert isinstance(run(exe, small[0], csi_file(tmp_path, good[:n]), "csi", small[1], small[2], 2), dict), n


def test_counts_past_the_end(exe, small, tmp_path):
    good = small[3]
    refused(exe, small, tmp_path, good[:12] + struct.pack("<i", len(good)) + good[16:], "l_aux")
    refused(exe, small, tmp_path, good[:12] + struct.pack("<i", -1) + good[16:], "l_aux")
    # the first bin of the first reference with bins: its n_chunk
    ms, d, aux, refs, tail = split_csi(good)
    o = 16 + len(aux) + 4
    for bins in refs:
        o += 4
        if bins:
            break
    bad = bytearray(good)
    bad[o + 12:o + 16] = struct.pack("<i", 1 << 20)
    refused(exe, small, tmp_path, bytes(bad), "n_chunk")
    bad[o + 12:o + 16] = struct.pack("<i", -2)
    refused(exe, small, tmp_path, bytes(bad), "n_chunk")


def test_reference_count_must_match_the_header(exe, small, tmp_path):
    n = small[2]
    msg = refused(exe, small, tmp_path, small[3], "references", n_ref=n + 1)
    assert f"{n} references, the BAM header has {n + 1}" in msg
    refused(exe, small, tmp_path, small[3], "references", n_ref=n - 1)


def test_binning_that_overflows(exe, small, tmp_path):
    good = small[3]
    for ms, d in ((14, 10), (14, -1), (-1, 5), (60, 2), (1 << 30, 5)):
        refused(exe, small, tmp_path, good[:4] + struct.pack("<ii", ms, d) + good[12:], "overflows")
    # the deepest binning accepted reads (every bin is then an ordinary bin: the pseudo-bin of depth 9 is not in the payload)
    bam, first, n, _ = small
    res = run(exe, bam, csi_file(tmp_path, good[:4] + struct.pack("<ii", 14, 9) + good[12:]), "csi", first, n, 2)
    assert isinstance(res, dict) and not any(r[0] for r in res["ref"])
