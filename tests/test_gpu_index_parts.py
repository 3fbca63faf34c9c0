"""A BAM without an index cut between engines (NGSQ_F_INDEX_PART, ngsq_find_record, ngsq_join_bai; DESIGN.md section 4 K13
and section 5): the record anchor finder must return the first record start of its window, the joined .bai must be the one
engine's and the oracle's byte for byte wherever the file is cut, order violations at a cut must fail as one engine fails,
a decoy anchor must be refuted by the range in front of it, and qc integers over parts must be the oracle's.  The host
driver's `index --cuda-devices` and `qc --cuda-build-index` write the same bytes."""
import bisect
import os
import subprocess

import numpy as np
import pytest

from baiutil import bgzf_offsets, micro_bams, oracle_bai, oracle_keys, placed_minus_one_bam, unsorted_bams
from bamutil import rec, record, write_bam
from helpers import assert_same_ints, canonical_results, collect, merge_ints, oracle_ints

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "ngs_b200", "ngs-cuda-qc")
GC_SEED = 5
GRCH38 = "GRCh38_no_alt_AnalysisSet"


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _u8(bam):
    return np.ascontiguousarray(np.frombuffer(bam, dtype=np.uint8) if isinstance(bam, (bytes, bytearray)) else bam)


def _refs(hdr):
    from ngs_b200 import formats
    return [l for _, l in hdr.refs], [1 if formats.is_primary(n) else 0 for n, _ in hdr.refs]


def find_from(eng, bam, coff, blocks=1):
    """The finder over a window of `blocks` blocks from file offset coff, doubled until it sees a record or reaches EOF."""
    from ngs_b200 import ffi
    b = _u8(bam)
    while True:
        arr, n, used = ffi.bgzf_walk(b[coff:coff + (blocks << 16)], coff)
        n = min(n, blocks)
        used = arr[n - 1].coffset + arr[n - 1].csize - coff if n else 0
        v, r = eng.find_record(np.ascontiguousarray(b[coff:coff + used]), coff)
        if v or coff + used >= b.size:
            return v, r
        blocks *= 2


def run_parts(bam, cuts, flags=None, engines=None, launch_blocks=0, split=()):
    """One NGSQ_F_INDEX_PART engine per range [first record, cut 1), [cut 1, cut 2), .., [last cut, EOF); returns the
    engines (finished) in file order."""
    from ngs_b200 import ffi, formats
    b = _u8(bam)
    if flags is None:
        flags = ffi.NGSQ_F_INDEX_PART | ffi.NGSQ_F_VERIFY_CRC
    bounds = None
    engines = list(engines or [])
    while len(engines) < len(cuts) + 1:
        engines.append(ffi.Engine(0, flags=flags, gc_seed=GC_SEED, launch_blocks=launch_blocks))
    hdr = formats.read_header(engines[0], b)
    bounds = [hdr.first_voffset] + list(cuts)
    blocks, nb, _ = ffi.bgzf_walk(b)
    lens, enabled = _refs(hdr)
    for i, first in enumerate(bounds):
        e = engines[i]
        e.reset()
        e.set_references(lens, enabled)
        for c in split:
            e.split_reference(c)
        end = bounds[i + 1] if i + 1 < len(bounds) else 0
        lo, hi = formats.shard_byte_range(formats.Shard(first, end, []), blocks, nb, b.size)
        e.set_range(first, end)
        e.submit(np.ascontiguousarray(b[lo:hi]), lo)
        e.finish()
    return engines[:len(bounds)]


def joined(bam, cuts, **kw):
    from ngs_b200 import ffi
    return ffi.join_bai(run_parts(bam, cuts, **kw))


def even_cuts(eng, bam, k):
    """k - 1 cuts the way the driver's planner takes them: targets snapped to the next block start, moved to the first
    record the finder sees; repeated anchors dropped.  Returns (cuts, reference ids of the records there)."""
    b = _u8(bam)
    from ngs_b200 import formats
    hdr = formats.read_header(eng, b)
    starts = [c for c, _, _ in bgzf_offsets(b)]
    base = hdr.first_voffset >> 16
    cuts, refs = [], []
    for j in range(1, k):
        t = base + (b.size - base) * j // k
        p = next((c for c in starts if c >= t), None)
        if p is None:
            continue
        v, r = find_from(eng, b, p, 4)
        if v and v > (cuts[-1] if cuts else hdr.first_voffset):
            cuts.append(v)
            refs.append(r)
    return cuts, refs


def _finder_engine(bam):
    from ngs_b200 import ffi, formats
    eng = ffi.Engine(0, flags=ffi.NGSQ_F_INDEX_PART)
    hdr = formats.read_header(eng, _u8(bam))
    eng.set_references(*_refs(hdr))
    return eng, hdr


_SYNTH = {}


def _synth(shape, level):
    from ngs_b200 import ffi
    if (shape, level) not in _SYNTH:
        bam, bai, info = ffi.synth_bam(shape, 1500 if shape == 2 else 40000, level=level)
        _SYNTH[(shape, level)] = (bam, bai, info, oracle_bai(bam))
    return _SYNTH[(shape, level)]


# ---------------------------------------------------------------- the finder
@pytest.mark.parametrize("level", [1, 6])
@pytest.mark.parametrize("shape", [0, 1, 2, 3])
def test_finder_returns_the_first_record_start_of_every_block(shape, level):
    bam, _, _, _ = _synth(shape, level)
    keys, err = oracle_keys(bam)
    assert err is None
    starts = sorted(k[7] for k in keys)
    eng, hdr = _finder_engine(bam)
    b = _u8(bam)
    empty_windows = 0
    for coff, _, isize in bgzf_offsets(b):
        if coff < hdr.first_voffset >> 16 or not isize:
            continue
        i = bisect.bisect_left(starts, coff << 16)
        want = starts[i] if i < len(starts) else 0
        v, r = find_from(eng, b, coff)
        assert v == want, (coff, v, want)
        if v:
            assert r == keys[i][0]
        # one block alone: its first record start, or 0 when the block lies inside one record (or the start is too close
        # to the block's end for a header to fit)
        one, _ = eng.find_record(np.ascontiguousarray(b[coff:coff + int.from_bytes(b[coff + 16:coff + 18].tobytes(), "little") + 1]), coff)
        assert one in (0, want)
        empty_windows += one == 0
    if shape == 2:
        assert empty_windows > 0  # blocks inside long reads


def test_finder_needs_the_references_and_whole_blocks():
    from ngs_b200 import ffi
    bam, _, _, _ = _synth(0, 1)
    eng = ffi.Engine(0, flags=ffi.NGSQ_F_INDEX_PART)
    b = _u8(bam)
    with pytest.raises(ffi.NgsqError, match="ngsq_set_references") as ex:
        eng.find_record(np.ascontiguousarray(b[:1000]), 0)
    assert ex.value.code == -1
    eng, _ = _finder_engine(bam)
    with pytest.raises(ffi.NgsqError) as ex:
        eng.find_record(np.ascontiguousarray(b[:1000]), 0)  # ends inside a block
    assert ex.value.code == -3


# ---------------------------------------------------------------- byte identity
@pytest.mark.parametrize("k", [2, 3, 5, 8])
@pytest.mark.parametrize("level", [1, 6])
@pytest.mark.parametrize("shape", [0, 1, 2, 3])
def test_joined_bai_equals_one_engine_and_the_oracle(shape, level, k):
    from test_gpu_index import gpu_bai
    bam, _, _, want = _synth(shape, level)
    eng, _ = _finder_engine(bam)
    cuts, _ = even_cuts(eng, bam, k)
    assert len(cuts) == k - 1
    assert joined(bam, cuts, launch_blocks=5) == gpu_bai(bam)[0] == want


@pytest.mark.parametrize("name", sorted(micro_bams()) + ["placed_minus_one"])
def test_micro_bams_cut_at_every_block_start(name):
    """One cut at every block start (the first record at or after it), then all of them at once: runs crossing a cut, a
    cut in the unplaced tail, the overhang list across a cut, a cut inside a record."""
    bam = placed_minus_one_bam()[0] if name == "placed_minus_one" else micro_bams()[name][0]
    want = oracle_bai(bam)
    keys, _ = oracle_keys(bam)
    starts = sorted(k[7] for k in keys)
    b = _u8(bam)
    eng, hdr = _finder_engine(bam)
    cuts = []
    for coff, _, isize in bgzf_offsets(b):
        if coff <= hdr.first_voffset >> 16 or not isize:
            continue
        v, _ = find_from(eng, b, coff)
        assert v == next((s for s in starts if s >= coff << 16), 0)
        if v and v > hdr.first_voffset and v not in cuts:
            cuts.append(v)
    pool = []
    for v in cuts:
        pool = run_parts(bam, [v], engines=pool)
        from ngs_b200 import ffi
        assert ffi.join_bai(pool) == want, v
    if cuts:
        assert joined(bam, cuts) == want


# ---------------------------------------------------------------- order across a cut
@pytest.mark.parametrize("name", sorted(unsorted_bams()))
def test_unsorted_at_a_cut_fails_like_one_engine(name):
    from ngs_b200 import ffi
    bam, first_bad = unsorted_bams()[name]
    keys, _ = oracle_keys(bam)
    bad = keys[first_bad][7]
    parts = run_parts(bam, [bad])
    assert parts[1].stats()["records"] == len(keys) - first_bad
    with pytest.raises(ffi.NgsqError, match=f"virtual offset {bad} ") as ex:
        ffi.join_bai(parts)
    assert ex.value.code == -14
    # the same violation inside a part: the part's own check, the same message
    with pytest.raises(ffi.NgsqError, match=f"virtual offset {bad} ") as ex:
        ffi.join_bai(run_parts(bam, []))
    assert ex.value.code == -14


# ---------------------------------------------------------------- a decoy anchor at a cut
REFS = [("chr1", 100000), ("chr2", 50000)]


def decoy_case():
    """test_gpu_decoy.py's construction, with the fake records ending exactly where their host record ends, so that their
    chain runs on into the true records and the finder takes them; the decoy starts the first block behind the middle of
    the file (the driver's cut on two devices): the records in front of it are random, the ones behind it compress well."""
    fake = b"".join(record(name="d", flag=0, ref=0, pos=5 + i, mapq=30, cigar="10M", seq="ACGTACGTAC", qual=[30] * 10) for i in range(3))
    rng = np.random.default_rng(3)
    before = [rec(name=f"a{i}", flag=0x43, ref=0, pos=100 + i, next_ref=0, next_pos=300, tlen=250, mapq=30, cigar="50M",
                  seq="".join(rng.choice(list("ACGT"), 50)), qual=[int(q) for q in rng.integers(2, 40, 50)]) for i in range(300)]
    host = rec(name="host", flag=0x83, ref=0, pos=500, next_ref=0, next_pos=100, tlen=-450, mapq=30, cigar="50M", seq="TTGCA" * 10,
               qual=[35] * 50, aux=fake)
    after = [rec(name=f"b{i}", flag=0x43, ref=1, pos=10 + 9 * i, next_ref=0, next_pos=7, mapq=30, cigar="20M5D30M", seq="GGCAT" * 10,
                 qual=[20] * 50) for i in range(60)]
    cut = sum(len(r[0]) for r in before) + len(host[0]) - len(fake)
    bam, bai = write_bam(REFS, before + [host] + after, block_payload=[cut, 0xFF00])
    return _u8(bam), fake


def test_the_decoy_is_found_and_the_part_in_front_of_it_fails():
    from ngs_b200 import ffi
    bam, fake = decoy_case()
    blocks = [c for c, _, isize in bgzf_offsets(bam) if isize]
    decoy_block = blocks[2]
    eng, hdr = _finder_engine(bam)
    v, r = find_from(eng, bam, decoy_block)
    assert v == decoy_block << 16 and r == 0  # the decoy, not the next true record
    keys, _ = oracle_keys(bam)
    assert v not in {k[7] for k in keys}
    with pytest.raises(ffi.NgsqError) as ex:
        run_parts(bam, [v])
    assert ex.value.code in (-8, -3)


def test_driver_recovers_from_the_decoy(tmp_path):
    bam, _ = decoy_case()
    hdr_block = bgzf_offsets(bam)[1][0]
    target = hdr_block + (bam.size - hdr_block) // 2
    assert next(c for c, _, _ in bgzf_offsets(bam) if c >= target) == [c for c, _, i in bgzf_offsets(bam) if i][2]
    p = str(tmp_path / "d.bam")
    bam.tofile(p)
    r = subprocess.run([DRIVER, "index", p, "--cuda-devices", "0,0"], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "not a record start" in r.stderr
    assert open(p + ".bai", "rb").read() == oracle_bai(bam)


# ---------------------------------------------------------------- argument errors
def test_argument_errors():
    from ngs_b200 import ffi
    with pytest.raises(ffi.NgsqError, match="instead of") as ex:
        ffi.Engine(0, flags=ffi.NGSQ_F_INDEX | ffi.NGSQ_F_INDEX_PART)
    assert ex.value.code == -1
    with pytest.raises(ffi.NgsqError, match="max_records") as ex:
        ffi.Engine(0, flags=ffi.NGSQ_F_INDEX_PART, max_records=5)
    assert ex.value.code == -1
    bam, _, _, _ = _synth(0, 1)
    eng, _ = _finder_engine(bam)
    cuts, _ = even_cuts(eng, bam, 3)
    parts = run_parts(bam, cuts)
    with pytest.raises(ffi.NgsqError, match="ngsq_join_bai") as ex:
        parts[0].bai()
    assert ex.value.code == -1

    def refused(ps, match):
        with pytest.raises(ffi.NgsqError, match=match) as ex:
            ffi.join_bai(ps)
        assert ex.value.code == -1
    refused([parts[0], parts[2]], "contiguous")
    refused([parts[1], parts[0], parts[2]], "contiguous")
    refused(parts[:2], "end of the data")
    whole = ffi.Engine(0, flags=ffi.NGSQ_F_INDEX)
    refused([whole], "NGSQ_F_INDEX_PART")
    fresh = ffi.Engine(0, flags=ffi.NGSQ_F_INDEX_PART)
    refused([fresh], "did not finish")
    other = run_parts(_synth(3, 1)[0], [])
    refused([parts[0], parts[1], other[0]], "references|contiguous")
    # a failed part is not joined
    bad = run_parts(bam, [cuts[0]])
    bad[0].reset()
    bad[0].set_range(0, 0)
    refused(bad, "did not finish|contiguous")
    # reduce and split references are allowed on a part (single rank: reduce needs a communicator)
    with pytest.raises(ffi.NgsqError) as ex:
        parts[0].reduce(0)
    assert ex.value.code == -9


# ---------------------------------------------------------------- qc over parts
@pytest.mark.parametrize("k", [2, 3, 5])
@pytest.mark.parametrize("shape", [0, 2, 3])
def test_qc_integers_over_parts_equal_the_oracle(shape, k):
    from ngs_b200 import ffi, formats
    from test_gpu_split import merge_split
    bam, bai, info, want_bai = _synth(shape, 1)
    want = oracle_ints(bam, bai, gc_seed=GC_SEED)
    eng, hdr = _finder_engine(bam)
    cuts, refs = even_cuts(eng, bam, k)
    split = sorted({r for r in refs if r >= 0})
    flags = ffi.NGSQ_F_INDEX_PART | ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_COVERAGE | ffi.NGSQ_F_VERIFY_CRC
    parts = run_parts(bam, cuts, flags=flags, split=split)
    assert ffi.join_bai(parts) == want_bai
    merge_split(parts, split, 0)
    lens, enabled = _refs(hdr)
    got = merge_ints([collect(e, lens, enabled) for e in parts])
    assert sum(e.stats()["records"] for e in parts) == info["n_records"]
    assert_same_ints(got, want)


# ---------------------------------------------------------------- host driver
def _run(args):
    return subprocess.run([DRIVER] + args, capture_output=True, text=True)


def test_driver_index_on_repeated_devices(tmp_path):
    bam, _, _, want = _synth(1, 6)
    p = str(tmp_path / "s.bam")
    bam.tofile(p)
    r = _run(["index", p, "--cuda-devices", "0,0,0", "--cuda-chunk-mb", "1"])
    assert r.returncode == 0, r.stderr
    assert "3 parts" in r.stderr
    got = open(p + ".bai", "rb").read()
    assert got == want
    before = os.stat(p + ".bai").st_mtime_ns
    r = _run(["index", p, "--cuda-devices", "0,0"])
    assert r.returncode != 0 and "exists" in r.stderr
    assert open(p + ".bai", "rb").read() == got and os.stat(p + ".bai").st_mtime_ns == before


def test_driver_qc_build_index(tmp_path):
    bam, bai, _, want_bai = _synth(3, 1)
    p = str(tmp_path / "q.bam")
    bam.tofile(p)
    r = _run(["qc", p, GRCH38, "-o", str(tmp_path), "-p", "built", "--cuda-gc-seed", "4"])
    assert r.returncode != 0 and "index" in r.stderr.lower()  # without the flag a missing .bai is an error, as before
    r = _run(["qc", p, GRCH38, "-o", str(tmp_path), "-p", "built", "--cuda-gc-seed", "4", "--cuda-build-index"])
    assert r.returncode == 0, r.stderr
    assert open(p + ".bai", "rb").read() == want_bai
    oracle_ints(bam, bai, gc_seed=4, json_path=str(tmp_path / "o.json"))
    assert canonical_results(str(tmp_path / "built.results.json")) == canonical_results(str(tmp_path / "o.json"))
    # an existing index is read and left as it is
    before = os.stat(p + ".bai").st_mtime_ns
    r = _run(["qc", p, GRCH38, "-o", str(tmp_path), "-p", "again", "--cuda-gc-seed", "4", "--cuda-build-index"])
    assert r.returncode == 0, r.stderr
    assert os.stat(p + ".bai").st_mtime_ns == before
    assert canonical_results(str(tmp_path / "again.results.json")) == canonical_results(str(tmp_path / "o.json"))
    r = _run(["qc", p, GRCH38, "-o", str(tmp_path), "-p", "n", "-n", "100", "--cuda-build-index"])
    assert r.returncode != 0 and "-n" in r.stderr


@pytest.mark.parametrize("devices", ["0", "0,0"])
def test_driver_unsorted_input_writes_no_index(tmp_path, devices):
    bam, _ = unsorted_bams()["position"]
    p = str(tmp_path / "u.bam")
    open(p, "wb").write(bytes(bam))
    if devices == "0":
        r = _run(["qc", p, GRCH38, "-o", str(tmp_path), "--cuda-build-index"])
    else:
        r = _run(["index", p, "--cuda-devices", devices])
    assert r.returncode != 0 and "not coordinate-sorted" in r.stderr
    assert not os.path.exists(p + ".bai")


@pytest.mark.parametrize("n", [2, 4])
def test_driver_on_distinct_devices(tmp_path, n):
    if _n_gpus() < n:
        pytest.skip(f"needs {n} GPUs")
    devs = ",".join(str(i) for i in range(n))
    bam, bai, _, want_bai = _synth(0, 1)
    p, q = str(tmp_path / "i.bam"), str(tmp_path / "q.bam")
    bam.tofile(p)
    bam.tofile(q)
    r = _run(["index", p, "--cuda-devices", devs])
    assert r.returncode == 0, r.stderr
    assert open(p + ".bai", "rb").read() == want_bai
    r = _run(["qc", q, GRCH38, "-o", str(tmp_path), "-p", "multi", "--cuda-gc-seed", "4", "--cuda-devices", devs, "--cuda-build-index"])
    assert r.returncode == 0, r.stderr
    assert open(q + ".bai", "rb").read() == want_bai
    oracle_ints(bam, bai, gc_seed=4, json_path=str(tmp_path / "o.json"))
    assert canonical_results(str(tmp_path / "multi.results.json")) == canonical_results(str(tmp_path / "o.json"))
