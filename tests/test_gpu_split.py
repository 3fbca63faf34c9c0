"""Shards cut inside contigs (DESIGN.md section 5): k engines, each over one shard of plan_shards_split, declare the split
references, and their partial arrays are summed into a root engine's (here with torch, the way a caller with its own
collective does) before ngsq_resolve_split.  Every integer must equal the oracle's over the whole file, the GC window
histogram included (windows are keyed by the records' virtual offsets, which do not change with the cut).  The multi-GPU
tests at the end run the same merge through ngsq_reduce and the host driver."""
import os
import subprocess
import threading

import numpy as np
import pytest

from bamutil import rec, write_bam
from helpers import assert_same_ints, canonical_results, collect, merge_ints, oracle_ints

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "ngs_b200", "ngs-cuda-qc")
GC_SEED = 5


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _view(ptr, n, typestr):
    """A torch tensor over device memory the engine owns (zero-copy, through __cuda_array_interface__)."""
    import torch

    class _Mem:
        __cuda_array_interface__ = {"shape": (int(n),), "typestr": typestr, "data": (int(ptr), False), "version": 3}
    return torch.as_tensor(_Mem(), device="cuda")


# (pointer, length, dtype for the sum): the u32 / u64 counters are summed through same-width signed views (wrap-around adds)
_ARRAYS = [("diff", "n_diff", "<i4"), ("tile_sums", "n_tiles", "<i4"), ("touched", None, "<i8"),
           ("edit_refs", "n_positions", "<i4"), ("edit_alts", "n_positions", "<i4")]


def merge_split(engines, split, root):
    import torch
    for c in split:
        arrs = [e.split_arrays(c) for e in engines]
        for key, n_key, typ in _ARRAYS:
            if not arrs[root][key]:
                continue
            n = arrs[root][n_key] if n_key else 1
            dst = _view(arrs[root][key], n, typ)
            for i, a in enumerate(arrs):
                if i != root:
                    dst += _view(a[key], n, typ)
    torch.cuda.synchronize()
    for i, e in enumerate(engines):
        e.resolve_split(i == root)


def run_split(bam, bai, k, flags=None, fasta=None, root=None):
    """k engines on device 0, one per shard of plan_shards_split; returns (engines, header, shards, split, root) after
    every engine finished, before the merge.  root=None picks an engine that holds no records of some split reference
    when there is one (the root must resolve what only other ranks touched)."""
    from ngs_b200 import ffi, formats
    b = np.ascontiguousarray(bam)
    flags = flags if flags is not None else ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_COVERAGE | ffi.NGSQ_F_VERIFY_CRC
    engines = [ffi.Engine(0, flags=flags, gc_seed=GC_SEED) for _ in range(k)]
    hdr = formats.read_header(engines[0], b)
    shards, split = formats.plan_shards_split(hdr, formats.parse_bai(bytes(np.asarray(bai))), k, b.size)
    blocks, nb, _ = ffi.bgzf_walk(b)
    lens = [l for _, l in hdr.refs]
    enabled = [1 if formats.is_primary(n) else 0 for n, _ in hdr.refs]
    for e, s in zip(engines, shards):
        e.set_references(lens, enabled)
        for c, (name, _) in enumerate(hdr.refs):
            if fasta and name in fasta:
                e.set_reference_bases(c, fasta[name])
        for c in split:
            e.split_reference(c)
        if s.first_voffset == 0 and not s.contigs:  # no anchor left for this engine
            e.set_range(0, 0)
        else:
            lo, hi = formats.shard_byte_range(s, blocks, nb, b.size)
            e.set_range(s.first_voffset, s.end_voffset)
            e.submit(np.ascontiguousarray(b[lo:hi]), lo)
        e.finish()
    if root is None:
        root = next((i for i, s in enumerate(shards) if any(c not in s.contigs for c in split)), 0)
    return engines, hdr, shards, split, root


def split_ints(bam, bai, k):
    from ngs_b200 import ffi, formats
    engines, hdr, shards, split, root = run_split(bam, bai, k)
    lens = [l for _, l in hdr.refs]
    enabled = [1 if formats.is_primary(n) else 0 for n, _ in hdr.refs]
    for c in split:  # partial numbers are refused until the merge
        with pytest.raises(ffi.NgsqError) as ei:
            engines[root].coverage_contig(c, lens[c])
        assert ei.value.code == -1
    merge_split(engines, split, root)
    parts = [collect(e, lens, enabled) for e in engines]
    for c in split:  # the root alone holds a split contig's numbers
        assert all(c not in p["coverage"] for i, p in enumerate(parts) if i != root)
    got = merge_ints(parts)
    got["records"] = sum(p["stats"]["records"] for p in parts)
    return got, split, shards, root


_ORACLE = {}


def _synth(shape, level):
    from ngs_b200 import ffi
    key = (shape, level)
    if key not in _ORACLE:
        bam, bai, info = ffi.synth_bam(shape, 4000 if shape == 2 else 60000, level=level)
        _ORACLE[key] = (bam, bai, info, oracle_ints(bam, bai, gc_seed=GC_SEED))
    return _ORACLE[key]


@pytest.mark.parametrize("k", [2, 3, 5])
@pytest.mark.parametrize("level", [1, 6])
@pytest.mark.parametrize("shape", [0, 2, 3])
def test_split_shards_equal_the_whole_file(shape, level, k):
    bam, bai, info, want = _synth(shape, level)
    got, split, shards, root = split_ints(bam, bai, k)
    assert got["records"] == info["n_records"]
    assert_same_ints(got, want)


def test_root_without_records_of_a_split_contig():
    """Shape 0 over 5 shards: chr1 is cut, and the root holds none of its records."""
    bam, bai, info, want = _synth(0, 1)
    engines, hdr, shards, split, root = run_split(bam, bai, 5)
    assert any(c not in shards[root].contigs for c in split)
    got, split2, _, root2 = split_ints(bam, bai, 5)
    assert root2 == root and split2 == split
    assert_same_ints(got, want)


# ---- hand-built single-contig files
L1 = 400_000


def _dense(lo, hi, step, cigar="100M", seq_len=100, name="d"):
    n = seq_len
    return [rec(name=f"{name}{p}", flag=0, ref=0, pos=p, mapq=60, cigar=cigar, seq="ACGT" * (n // 4), qual=[30] * n)
            for p in range(lo, hi, step)]


def _file_overhang():
    """Short reads every 37 bases: every cut has reads overhanging it; reads past the contig end close the file."""
    r = _dense(0, L1 - 120, 37)
    r += [rec(name=f"past{i}", flag=0, ref=0, pos=L1 - 60 + i, mapq=60, cigar="100M", seq="ACGT" * 25, qual=[30] * 100) for i in range(5)]
    return r


def _file_deep_pile():
    """Records of 16 kb without bases, one every 5 positions over half the contig: depth 3200 > 2048 at every cut."""
    return [rec(name=f"p{i}", flag=0, ref=0, pos=5 * i, mapq=60, cigar="16000M") for i in range(40_000)]


def _file_star_cigar_at_cuts():
    """Every 16 kb window starts with a placed `*`-CIGAR record and no read crosses a window start, so every anchor, and
    every cut, is a `*`-CIGAR record; a 50 kb bin straddles most cuts."""
    r = []
    for w in range(L1 // 16384):
        base = w * 16384
        r.append(rec(name=f"s{w}", flag=0, ref=0, pos=base, mapq=60, cigar="*", seq="ACGT", qual=[30] * 4))
        r += _dense(base + 50, base + 16384 - 200, 160, name=f"w{w}_")
    return r


HAND = {"overhang": _file_overhang, "deep_pile": _file_deep_pile, "star_cigar": _file_star_cigar_at_cuts}


@pytest.mark.parametrize("k", [2, 3, 5])
@pytest.mark.parametrize("name", sorted(HAND))
def test_hand_built_single_contig(name, k):
    recs = HAND[name]()
    recs.append(rec(name="unplaced", flag=4, seq="ACGT", qual=[30] * 4))
    bam, bai = write_bam([("chr1", L1)], recs, level=1)
    b, x = np.frombuffer(bam, dtype=np.uint8).copy(), np.frombuffer(bai, dtype=np.uint8).copy()
    want = oracle_ints(b, x, gc_seed=GC_SEED)
    got, split, shards, root = split_ints(b, x, k)
    assert split == [0]
    assert len([s for s in shards if s.contigs]) == k
    assert_same_ints(got, want)


# ---- Edits: the VAF histogram and the per-position counters of a split contig
def _edits_case(refs=(("chr1", 70_000),), seed=23):
    """Reads every 41 bases with up to three substitutions each, over every contig of `refs` (header order)."""
    rng = np.random.default_rng(seed)
    fasta, recs = {}, []
    for c, (name, L) in enumerate(refs):
        ref = "".join(rng.choice(list("ACGT"), size=L))
        fasta[name] = ref.encode()
        for p in range(0, L - 200, 41):
            n = 60
            s = list(ref[p:p + n])
            for j in rng.integers(0, n, size=int(rng.integers(0, 4))):
                s[j] = "A" if s[j] != "A" else "C"
            recs.append(rec(name=f"e{c}_{p}", flag=0, ref=c, pos=p, mapq=60, cigar=f"{n}M", seq="".join(s), qual=[30] * n))
    bam, bai = write_bam(list(refs), recs, level=1)
    return np.frombuffer(bam, dtype=np.uint8).copy(), np.frombuffer(bai, dtype=np.uint8).copy(), fasta, refs[0][1]


@pytest.mark.parametrize("k", [2, 3])
def test_edits_of_split_contig_equal_one_engine(k):
    from ngs_b200 import ffi
    bam, bai, fasta, L = _edits_case()
    flags = ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_COVERAGE | ffi.NGSQ_F_VERIFY_CRC | ffi.NGSQ_F_EDITS
    whole, _, _, _, _ = run_split(bam, bai, 1, flags=flags, fasta=fasta)
    one, two, vaf, n = whole[0].edits()
    refs, alts = whole[0].edit_positions(0, L)
    assert vaf.sum() > 0
    engines, hdr, shards, split, root = run_split(bam, bai, k, flags=flags, fasta=fasta)
    assert split == [0]
    for e in engines:  # incomplete before the merge
        for call in (lambda: e.edits(), lambda: e.edit_positions(0, L)):
            with pytest.raises(ffi.NgsqError) as ei:
                call()
            assert ei.value.code == -1
    merge_split(engines, split, root)
    got = [e.edits() for e in engines]
    np.testing.assert_array_equal(sum(g[0] for g in got), one)
    np.testing.assert_array_equal(sum(g[1] for g in got), two)
    np.testing.assert_array_equal(sum(g[2] for g in got), vaf)
    assert sum(g[3] for g in got) == n
    pos = [e.edit_positions(0, L) for e in engines]
    np.testing.assert_array_equal(pos[root][0], refs)
    np.testing.assert_array_equal(pos[root][1], alts)
    for i, (r, a) in enumerate(pos):
        if i != root:
            assert not r.any() and not a.any()


@pytest.mark.parametrize("k", [2, 3])
def test_edits_of_split_contig_between_whole_contigs(k):
    """chr1 is cut, chr2 before it and chrM after it are whole: the VAF pass of ngsq_finish runs over the runs of whole
    contigs on each side, the root's over chr1 after the merge."""
    from ngs_b200 import ffi
    refs = (("chr2", 8_000), ("chr1", 70_000), ("chrM", 5_000))
    bam, bai, fasta, _ = _edits_case(refs, seed=29)
    flags = ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_COVERAGE | ffi.NGSQ_F_VERIFY_CRC | ffi.NGSQ_F_EDITS
    whole, _, _, _, _ = run_split(bam, bai, 1, flags=flags, fasta=fasta)
    one, two, vaf, n = whole[0].edits()
    want = [whole[0].edit_positions(c, L) for c, (_, L) in enumerate(refs)]
    engines, hdr, shards, split, root = run_split(bam, bai, k, flags=flags, fasta=fasta)
    assert split == [1]
    merge_split(engines, split, root)
    got = [e.edits() for e in engines]
    np.testing.assert_array_equal(sum(g[0] for g in got), one)
    np.testing.assert_array_equal(sum(g[1] for g in got), two)
    np.testing.assert_array_equal(sum(g[2] for g in got), vaf)
    assert sum(g[3] for g in got) == n and vaf.sum() > 0
    for c, (_, L) in enumerate(refs):
        pos = [e.edit_positions(c, L) for e in engines]
        np.testing.assert_array_equal(sum(p[0].astype(np.uint64) for p in pos), want[c][0])
        np.testing.assert_array_equal(sum(p[1].astype(np.uint64) for p in pos), want[c][1])


def test_split_reference_argument_errors():
    from ngs_b200 import ffi
    for kw in ({"flags": ffi.NGSQ_F_INDEX}, {"flags": ffi.NGSQ_F_COVERAGE, "max_records": 10}):
        e = ffi.Engine(0, **kw)
        e.set_references([1000], [1])
        with pytest.raises(ffi.NgsqError) as ei:
            e.split_reference(0)
        assert ei.value.code == -1
        e.close()
    e = ffi.Engine(0)
    with pytest.raises(ffi.NgsqError):
        e.split_reference(0)  # before ngsq_set_references
    e.set_references([1000, 2000], [1, 1])
    with pytest.raises(ffi.NgsqError):
        e.split_reference(2)
    with pytest.raises(ffi.NgsqError):
        e.split_arrays(1)  # not declared
    e.split_reference(1)
    a = e.split_arrays(1)
    assert a["n_diff"] == 2002 and a["n_tiles"] == 1 and a["diff"] and not a["edit_refs"]
    with pytest.raises(ffi.NgsqError):
        e.resolve_split(True)  # before finish
    e.close()


# ---- several GPUs: ngsq_reduce and the host driver
def _write(tmp_path, bam, bai, name):
    p = str(tmp_path / name)
    open(p, "wb").write(bytes(bam))
    open(p + ".bai", "wb").write(bytes(bai))
    return p


def _drive(args):
    r = subprocess.run([DRIVER] + args, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return r


@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs")
def test_driver_two_devices_single_contig(tmp_path):
    bam, bai, fasta, L = _edits_case()
    p = _write(tmp_path, bam, bai, "one.bam")
    fa = str(tmp_path / "ref.fa")
    open(fa, "wb").write(b">chr1\n" + fasta["chr1"] + b"\n")
    r = _drive(["qc", p, "GRCh38_no_alt_AnalysisSet", "-o", str(tmp_path), "-p", "two", "--cuda-devices", "0,1", "--cuda-gc-seed", "6"])
    assert "Sharding inside contigs" in r.stderr
    want_path = str(tmp_path / "o.json")
    oracle_ints(bam, bai, gc_seed=6, json_path=want_path)
    assert canonical_results(str(tmp_path / "two.results.json")) == canonical_results(want_path)
    for devs, tag in (("0", "v1"), ("0,1", "v2")):
        _drive(["qc", p, "GRCh38_no_alt_AnalysisSet", "-o", str(tmp_path), "-p", tag, "--cuda-devices", devs, "-r", fa,
                "--vaf-file", str(tmp_path / f"{tag}.vaf")])
    assert open(tmp_path / "v1.vaf", "rb").read() == open(tmp_path / "v2.vaf", "rb").read()
    assert canonical_results(str(tmp_path / "v1.results.json")) == canonical_results(str(tmp_path / "v2.results.json"))


@pytest.mark.skipif(_n_gpus() < 4, reason="needs four GPUs")
def test_driver_four_devices_shape0(tmp_path):
    from ngs_b200 import ffi
    bam, bai, info = ffi.synth_bam(0, 200000, level=1)
    p = _write(tmp_path, bam, bai, "s0.bam")
    r = _drive(["qc", p, "GRCh38_no_alt_AnalysisSet", "-o", str(tmp_path), "-p", "four", "--cuda-devices", "0,1,2,3", "--cuda-gc-seed", "6"])
    assert "Sharding inside contigs" in r.stderr
    want_path = str(tmp_path / "o.json")
    oracle_ints(bam, bai, gc_seed=6, json_path=want_path)
    assert canonical_results(str(tmp_path / "four.results.json")) == canonical_results(want_path)


def _two_rank_reduce(bam, bai, declare):
    """Two engines on devices 0 and 1 over the 2-shard split plan; declare(rank, split) -> references that rank declares.
    Returns each rank's exception (or None) from ngsq_reduce."""
    from ngs_b200 import ffi, formats
    b = np.ascontiguousarray(bam)
    engines = [ffi.Engine(d, flags=ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_COVERAGE, gc_seed=GC_SEED) for d in (0, 1)]
    hdr = formats.read_header(engines[0], b)
    shards, split = formats.plan_shards_split(hdr, formats.parse_bai(bytes(np.asarray(bai))), 2, b.size)
    blocks, nb, _ = ffi.bgzf_walk(b)
    uid = ffi.nccl_unique_id()
    errs = [None, None]

    def rank(i):
        try:
            e = engines[i]
            e.set_references([l for _, l in hdr.refs], [1 if formats.is_primary(n) else 0 for n, _ in hdr.refs])
            for c in declare(i, split):
                e.split_reference(c)
            lo, hi = formats.shard_byte_range(shards[i], blocks, nb, b.size)
            e.set_range(shards[i].first_voffset, shards[i].end_voffset)
            e.submit(np.ascontiguousarray(b[lo:hi]), lo)
            e.finish()
            e.comm_init(2, i, uid)
            e.reduce(0)
        except Exception as ex:  # noqa: BLE001
            errs[i] = ex
    ts = [threading.Thread(target=rank, args=(i,)) for i in (0, 1)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    return engines, hdr, errs


@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs")
def test_reduce_merges_and_checks_the_split_set():
    from ngs_b200 import formats
    bam, bai, info, want = _synth(0, 1)
    engines, hdr, errs = _two_rank_reduce(bam, bai, lambda i, split: split)
    assert errs == [None, None]
    lens = [l for _, l in hdr.refs]
    enabled = [1 if formats.is_primary(n) else 0 for n, _ in hdr.refs]
    assert_same_ints(collect(engines[0], lens, enabled), want)
    # different split sets: refused before any split array moves
    _, _, errs = _two_rank_reduce(bam, bai, lambda i, split: split if i == 0 else [])
    assert all(getattr(x, "code", None) == -1 for x in errs), errs
    # a contig cut across ranks without being declared fails as before
    _, _, errs = _two_rank_reduce(bam, bai, lambda i, split: [])
    assert all(x is not None and "holds coverage from 2 ranks" in str(x) for x in errs), errs
