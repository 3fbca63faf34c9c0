"""`qc --cuda-also` (DESIGN.md section 5, "Several files"): the records of a coordinate-sorted file S written as k files
(tests/splitutil.py: contiguous chunks, round-robin, random assignment; a header-only file, a one-record file and a file of
unmapped records) and checked as one sample.  The results equal S's, except the GC window of reads longer than 101 bases: it is
keyed by the record's virtual offset in its own file, so for those the GC histogram and nucleobase counts must equal the sum of
the oracle's record pass over each file.

On one device: the driver's JSON (and `--vaf-file`) against S's; at the ABI, ngsq_next_file against separate engines and the
oracle, its refusals, an empty file in a queue, a truncated file; the queue's rerun for a read longer than the quality table; a
decoy anchor in a cut file, part by part.  On several devices (skipped when the box has fewer): the driver against its
one-device run."""
import os
import subprocess

import numpy as np
import pytest

from bamutil import EOF_BLOCK, bgzf_block, rec, write_bam
from helpers import assert_same_ints, canonical_results, collect, engine_ints, oracle_ints
from orderutil import split_records
from splitutil import SPLITS, edge_files, split_bam

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "ngs_b200", "ngs-cuda-qc")
GRCH38 = "GRCh38_no_alt_AnalysisSet"
GC_SEED = 5
LONG_SHAPES = {0, 1, 2}  # 2x150 and long reads: GC windows keyed by virtual offset; shape 3 is 2x100


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


_S = {}


def _synth(shape):
    from ngs_b200 import ffi
    if shape not in _S:
        _S[shape] = ffi.synth_bam(shape, 20000, level=1)
    return _S[shape]


def _write(path, data):
    with open(path, "wb") as f:
        f.write(bytes(data))
    return str(path)


def _write_all(tmp_path, files, stem="f"):
    return [_write(tmp_path / f"{stem}{i}.bam", f) for i, f in enumerate(files)]


def _qc(paths, outdir, prefix, *extra):
    also = [a for p in paths[1:] for a in ("--cuda-also", p)]
    r = subprocess.run([DRIVER, "qc", paths[0], GRCH38, "-o", str(outdir), "-p", prefix, "--cuda-gc-seed", str(GC_SEED)] + also + list(extra),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return os.path.join(str(outdir), prefix + ".results.json"), r.stderr


def _s_json(tmp_path, shape):
    bam, bai, _ = _synth(shape)
    s = _write(tmp_path / "s.bam", bam)
    _write(s + ".bai", bai)
    return _qc([s], tmp_path, "s")[0]


def _summed_gc(files, s_bai):
    hist, nuc = 0, 0
    for f in files:
        o = oracle_ints(f, s_bai, gc_seed=GC_SEED, coverage=False)
        hist, nuc = hist + o["gc_hist"].astype(np.uint64), nuc + o["gc_nuc"].astype(np.uint64)
    return [int(x) for x in hist], [int(x) for x in nuc]


def assert_json_of_files(got_path, want_path, files, s_bai, gc_window):
    got, want = canonical_results(got_path), canonical_results(want_path)
    if gc_window:
        assert got == want
        return
    g, w = got.pop("gc_content"), want.pop("gc_content")
    assert got == want
    assert g["records"] == w["records"]
    hist, nuc = _summed_gc(files, s_bai)
    assert g["histogram"]["values"] == hist
    nb = g["nucleobases"]
    assert [nb["total_gc_count"], nb["total_at_count"], nb["total_other_count"]] == nuc


# ---------------------------------------------------------------- the driver on one device
@pytest.mark.parametrize("k", [2, 7])
@pytest.mark.parametrize("kind", SPLITS)
@pytest.mark.parametrize("shape", [3, 0])
def test_driver_json_of_the_files_equals_s(tmp_path, shape, kind, k):
    want = _s_json(tmp_path, shape)
    files = split_bam(_synth(shape)[0], k, kind, seed=7 + k)
    paths = _write_all(tmp_path, files)
    got, err = _qc(paths, tmp_path, "m")
    assert f"{k} files of one sample on one device" in err
    assert_json_of_files(got, want, files, _synth(shape)[1], gc_window=shape not in LONG_SHAPES)
    assert not any(os.path.exists(p + x) for p in paths for x in (".bai", ".csi"))


def test_driver_on_200_small_files_and_the_edge_files(tmp_path):
    """200 files of about 100 records (the per-file transition, many times), then a header-only file, a one-record file and
    a file of unmapped records in front of the rest; --cuda-any-order beside the flag changes nothing."""
    bam, bai, _ = _synth(3)
    want = _s_json(tmp_path, 3)
    paths = _write_all(tmp_path, split_bam(bam, 200, "contiguous", block_payload=0x1900), "c")
    got, err = _qc(paths, tmp_path, "many", "--cuda-perf")
    assert canonical_results(got) == canonical_results(want)
    import json
    perf = json.load(open(tmp_path / "many.perf.json"))
    assert [p["files"] for p in perf] == [200]
    paths = _write_all(tmp_path, edge_files(bam), "e")
    for extra in ([], ["--cuda-any-order"]):
        got, _ = _qc(paths, tmp_path, "edge", *extra)
        assert canonical_results(got) == canonical_results(want)
    got, _ = _qc(paths[1:] + paths[:1], tmp_path, "edge_last")  # the header-only file last
    assert canonical_results(got) == canonical_results(want)


def _edits_files(tmp_path):
    from test_oracle_edits import make_edits_case
    from test_oracle_features import gff_line
    bam, bai, fa, _, _ = make_edits_case(23)
    (tmp_path / "ref.fa").write_bytes(fa)
    (tmp_path / "m.gff").write_text("##gff-version 3\n" + gff_line("chr1", "gene", 200, 3000) + gff_line("chr1", "exon", 200, 700)
                                    + gff_line("chr1", "exon", 1500, 1900, "-") + gff_line("chr1", "five_prime_UTR", 200, 260)
                                    + gff_line("chr1", "CDS", 261, 700) + gff_line("chr2", "gene", 100, 2500)
                                    + gff_line("chr2", "three_prime_UTR", 2000, 2500) + gff_line("chrM", "gene", 1, 800))
    s = _write(tmp_path / "s.bam", bam)
    _write(s + ".bai", bai)
    return s, bam


@pytest.mark.parametrize("kind", SPLITS)
def test_driver_with_edits_vaf_file_and_features(tmp_path, kind):
    s, bam = _edits_files(tmp_path)
    opt = ["-r", str(tmp_path / "ref.fa"), "-f", str(tmp_path / "m.gff")]
    want, _ = _qc([s], tmp_path, "s", *opt, "--vaf-file", str(tmp_path / "s.vaf"))
    paths = _write_all(tmp_path, split_bam(bam, 3, kind, seed=2, block_payload=1700))
    got, _ = _qc(paths, tmp_path, "m", *opt, "--vaf-file", str(tmp_path / "m.vaf"))
    assert canonical_results(got) == canonical_results(want)
    doc = canonical_results(got)
    assert doc["edits"]["vaf_histogram"]["values"] and doc["features"]["records"]["processed"] > 0
    vaf = (tmp_path / "m.vaf").read_bytes()
    assert vaf == (tmp_path / "s.vaf").read_bytes() and vaf.count(b"\n") > 1000


def test_driver_refuses_a_different_dictionary_before_the_pass(tmp_path):
    bam = _synth(3)[0]
    hdr, recs = split_records(bam)
    from ngs_b200 import formats
    _, refs, _ = formats.parse_bam_header(hdr)
    from bamutil import header_bytes
    other = [(n, l + 1 if i == 2 else l) for i, (n, l) in enumerate(refs)]
    odd = bytes(bgzf_block(header_bytes(other), 1)) + EOF_BLOCK
    s = _write(tmp_path / "s.bam", bam)
    o = _write(tmp_path / "odd.bam", odd)
    r = subprocess.run([DRIVER, "qc", s, GRCH38, "--cuda-also", o, "-o", str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 1
    assert f"the reference sequences of {o} differ from those of {s}" in r.stderr and f"reference 2 is \"{refs[2][0]}\"" in r.stderr
    assert "Starting CUDA pass" not in r.stderr and not os.path.exists(tmp_path / "s.bam.results.json")


# ---------------------------------------------------------------- the ABI
def _flags(edits=False):
    from ngs_b200 import ffi
    return ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_COVERAGE | ffi.NGSQ_F_VERIFY_CRC | (ffi.NGSQ_F_EDITS if edits else 0)


def run_queue(files, engine=None, launch_blocks=5, fasta=None, split=False, skip_submit=()):
    """Every file through one engine, ngsq_next_file behind each (the files in skip_submit get a range and no chunk)."""
    from ngs_b200 import ffi, formats
    files = [np.ascontiguousarray(f) for f in files]
    e = engine or ffi.Engine(0, flags=_flags(fasta is not None), gc_seed=GC_SEED, launch_blocks=launch_blocks)
    hdrs = [formats.read_header(e, f) for f in files]
    lens = [l for _, l in hdrs[0].refs]
    enabled = [1 if formats.is_primary(n) else 0 for n, _ in hdrs[0].refs]
    e.set_references(lens, enabled)
    for c, (name, _) in enumerate(hdrs[0].refs):
        if fasta and name in fasta:
            e.set_reference_bases(c, fasta[name])
    if split:
        for c in range(len(lens)):
            e.split_reference(c)
    for i, (f, h) in enumerate(zip(files, hdrs)):
        e.set_range(h.first_voffset, 0)
        lo = h.first_voffset >> 16
        if i not in skip_submit and lo < f.size:
            e.submit(np.ascontiguousarray(f[lo:]), lo)
        e.next_file()
    e.finish()
    return e, lens, enabled


@pytest.mark.parametrize("shape", [3, 0])
def test_one_file_with_next_file_equals_the_plain_run(shape):
    bam = _synth(shape)[0]
    e, lens, enabled = run_queue([bam])
    got, want = collect(e, lens, enabled), engine_ints(bam, gc_seed=GC_SEED, launch_blocks=5)
    assert_same_ints(got, want)
    for k in ["records", "blocks", "compressed_bytes", "inflated_bytes", "max_read_len", "waves"]:
        assert got["stats"][k] == want["stats"][k], k


@pytest.mark.parametrize("shape", [3, 0])
def test_next_file_equals_separate_engines_and_the_oracle(shape):
    bam, bai, info = _synth(shape)
    files = split_bam(bam, 2, "round_robin")
    e, lens, enabled = run_queue(files)
    got = collect(e, lens, enabled)
    parts = [engine_ints(f, gc_seed=GC_SEED, launch_blocks=5) for f in files]
    for k in ["general", "tlen_hist", "gc_hist", "gc_nuc", "gc_rec"]:
        np.testing.assert_array_equal(got[k], parts[0][k] + parts[1][k], err_msg=k)
    for k in ["tlen_processed", "tlen_ignored"]:
        assert got[k] == parts[0][k] + parts[1][k]
    rows = max(p["quality"].shape[0] for p in parts)
    q = np.zeros((rows, 94), dtype=np.uint64)
    for p in parts:
        q[:p["quality"].shape[0]] += p["quality"]
    np.testing.assert_array_equal(got["quality"], q)
    st, ps = got["stats"], [p["stats"] for p in parts]
    for k in ["records", "blocks", "compressed_bytes", "inflated_bytes"]:
        assert st[k] == ps[0][k] + ps[1][k], k
    assert st["records"] == info["n_records"] and st["max_read_len"] == max(p["max_read_len"] for p in ps)
    want = oracle_ints(bam, bai, gc_seed=GC_SEED)
    assert_same_ints(got, want, gc_window=shape not in LONG_SHAPES)


def test_edits_of_the_queue_equal_separate_engines_and_s():
    from test_gpu_split import _edits_case
    refs = (("chr2", 8_000), ("chr1", 70_000), ("chrM", 5_000))
    bam, _, fasta, _ = _edits_case(refs, seed=29)
    files = split_bam(bam, 2, "random", seed=4, block_payload=2900)
    e, _, _ = run_queue(files, fasta=fasta)
    parts = [run_queue([f], fasta=fasta)[0] for f in files]
    whole = run_queue([bam], fasta=fasta)[0]
    one, two, vaf, n = e.edits()
    p = [x.edits() for x in parts]
    np.testing.assert_array_equal(one, p[0][0] + p[1][0])
    np.testing.assert_array_equal(two, p[0][1] + p[1][1])
    assert n == p[0][3] + p[1][3]
    np.testing.assert_array_equal(vaf, whole.edits()[2])
    assert vaf.sum() > 0
    for c, (_, L) in enumerate(refs):
        got, want = e.edit_positions(c, L), whole.edit_positions(c, L)
        np.testing.assert_array_equal(got[0], want[0])
        np.testing.assert_array_equal(got[1], want[1])


def test_an_empty_file_in_the_middle_of_a_queue():
    """Header-only files, and a file given a range but no chunk, contribute nothing."""
    bam, bai, info = _synth(3)
    want = oracle_ints(bam, bai, gc_seed=GC_SEED)
    files = edge_files(bam)  # header-only, one record, unmapped, two halves
    for order, skip in (([1, 0, 2, 3, 4], ()), ([3, 0, 0, 2, 1, 4, 0], ()), ([3, 1, 2, 4, 4], (4,))):
        e, lens, enabled = run_queue([files[i] for i in order], skip_submit=skip)
        got = collect(e, lens, enabled)
        assert got["stats"]["records"] == info["n_records"]
        assert_same_ints(got, want)


def test_next_file_refusals():
    from ngs_b200 import ffi
    bam = _synth(3)[0]

    def code(fn):
        with pytest.raises(ffi.NgsqError) as ex:
            fn()
        return ex.value.code

    e = ffi.Engine(0, flags=_flags(), gc_seed=GC_SEED)
    e.set_references([1000], [1])
    assert code(e.next_file) == -1  # before ngsq_set_range
    e.set_range(0, 0)
    e.next_file()
    assert code(e.next_file) == -1  # again before the next file's range
    assert code(lambda: e.submit(np.ascontiguousarray(bam), 0)) == -1  # a chunk before the next file's range
    e.finish()
    assert code(e.next_file) == -1  # after finish
    for flags in (ffi.NGSQ_F_INDEX, ffi.NGSQ_F_INDEX_PART, ffi.NGSQ_F_INDEX | ffi.NGSQ_F_INDEX_CSI):
        x = ffi.Engine(0, flags=flags)
        x.set_references([1000], [0])
        x.set_range(0, 0)
        assert code(x.next_file) == -1
    x = ffi.Engine(0, flags=_flags(), max_records=10)
    x.set_references([1000], [1])
    x.set_range(0, 0)
    assert code(x.next_file) == -1
    # the refused engine is unharmed: a reset run works
    e.reset()
    e2, lens, enabled = run_queue([bam], engine=e)
    assert collect(e2, lens, enabled)["stats"]["records"] == _synth(3)[2]["n_records"]


def test_a_file_that_ends_inside_a_record_fails_the_run():
    """The record open at the end of a file is not carried into the next one: the run fails as a truncated file does."""
    bam = _synth(3)[0]
    hdr, recs = split_records(bam)
    stream = b"".join(recs[:300])
    cut = bytes(bgzf_block(hdr, 1)) + bgzf_block(stream[:0x4000], 1) + bgzf_block(stream[0x4000:-17], 1) + EOF_BLOCK
    good = split_bam(bam, 2, "contiguous")[1]
    from ngs_b200 import ffi
    for files in ([cut, good], [good, cut]):
        with pytest.raises(ffi.NgsqError) as ex:
            run_queue([np.frombuffer(f, dtype=np.uint8) if isinstance(f, bytes) else f for f in files], launch_blocks=1)
        assert ex.value.code == -3, str(ex.value)


# ---------------------------------------------------------------- recovery paths
def _long_read_case():
    """S: short reads on chr1 and chr2 and one read of 131 073 bases on chr2, late in the file; the files: S cut in two."""
    rng = np.random.default_rng(9)
    refs = [("chr1", 400_000), ("chr2", 400_000)]
    recs = []
    for c in range(2):
        for i in range(1500):
            pos = 100 + 97 * i
            recs.append(rec(name=f"r{c}_{i}", flag=0, ref=c, pos=pos, mapq=60, cigar="100M",
                            seq="".join(rng.choice(list("ACGT"), 100)), qual=[int(q) for q in rng.integers(2, 41, 100)]))
        if c == 1:
            n = 131_073
            recs.append(rec(name="long", flag=0, ref=1, pos=200_000, mapq=60, cigar=f"{n}M",
                            seq="".join(rng.choice(list("ACGT"), n)), qual=[int(q) for q in rng.integers(2, 41, n)]))
    bam, bai = write_bam(refs, recs, level=1)
    return np.frombuffer(bam, dtype=np.uint8).copy(), np.frombuffer(bai, dtype=np.uint8).copy()


def test_a_read_longer_than_the_quality_table_reruns_the_queue(tmp_path):
    bam, bai = _long_read_case()
    files = split_bam(bam, 2, "contiguous", block_payload=0xFF00)
    s = _write(tmp_path / "s.bam", bam)
    _write(s + ".bai", bai)
    want, _ = _qc([s], tmp_path, "s")
    paths = _write_all(tmp_path, files)
    got, err = _qc(paths, tmp_path, "m")
    assert "enlarging the quality table and reading the files again" in err
    assert_json_of_files(got, want, files, bai, gc_window=False)
    # the queue's integers against the oracle over S (the engine that meets the long read is enlarged the same way)
    from ngs_b200 import ffi
    with pytest.raises(ffi.NgsqError) as ex:
        run_queue(files)
    assert ex.value.code == -13
    e = ffi.Engine(0, flags=_flags(), gc_seed=GC_SEED, launch_blocks=5, quality_positions=131_074)
    e, lens, enabled = run_queue(files, engine=e)
    o = oracle_ints(bam, bai, gc_seed=GC_SEED)
    assert_same_ints(collect(e, lens, enabled), o, gc_window=False)


def test_a_decoy_anchor_in_a_cut_file_is_recovered():
    """Fewer files than devices, part by part on one device: the decoy file cut at its decoy (the part in front fails with
    NGSQ_E_CHAIN or NGSQ_E_TRUNCATED; the driver's run_parts then runs it over both ranges and the next engine over an empty
    one), the second file whole on a third engine; every reference split and merged.  Equals one engine over both files."""
    from ngs_b200 import ffi
    from baiutil import bgzf_offsets
    from test_gpu_index_parts import _finder_engine, decoy_case, find_from
    from test_gpu_qc_any_order import merged_ints, run_cut
    from test_gpu_split import merge_split
    bam, _ = decoy_case()
    other = split_bam(bam, 2, "round_robin", block_payload=0x2100)[1]
    decoy_block = [c for c, _, isize in bgzf_offsets(bam) if isize][2]
    finder, _ = _finder_engine(bam)
    v, _ = find_from(finder, bam, decoy_block)
    assert v == decoy_block << 16
    engines = [ffi.Engine(0, flags=_flags(), gc_seed=GC_SEED, launch_blocks=5) for _ in range(3)]
    with pytest.raises(ffi.NgsqError) as ex:
        run_cut(bam, [v], engines=engines[:2])
    assert ex.value.code in (-8, -3)
    parts, lens, enabled = run_cut(bam, [None], engines=engines[:2])
    whole, _, _ = run_cut(other, [], engines=engines[2:])
    got = merged_ints(parts + whole, lens, enabled, root=2)
    q, _, _ = run_queue([bam, other], split=True)
    merge_split([q], list(range(len(lens))), 0)
    want = collect(q, lens, enabled)
    want["records"] = q.stats()["records"]
    assert got["records"] == want["records"]
    assert_same_ints(got, want)


# ---------------------------------------------------------------- several devices
@pytest.mark.parametrize("n", [2, 4])
def test_driver_on_several_devices_equals_one(tmp_path, n):
    if _n_gpus() < n:
        pytest.skip(f"needs {n} GPUs")
    devs = ",".join(str(i) for i in range(n))
    for shape in (1, 3):
        for k in sorted({7, n - 1} - {1}):  # F >= D, and F < D where two files fit
            paths = _write_all(tmp_path, split_bam(_synth(shape)[0], k, "random", seed=k), f"s{shape}k{k}_")
            one, _ = _qc(paths, tmp_path, f"one{shape}_{k}")
            many, err = _qc(paths, tmp_path, f"many{shape}_{k}", "--cuda-devices", devs)
            assert ("each cut between its devices" if k < n else "whole files queued on the devices") in err
            assert canonical_results(many) == canonical_results(one)
    s, bam = _edits_files(tmp_path)
    opt = ["-r", str(tmp_path / "ref.fa"), "-f", str(tmp_path / "m.gff")]
    for k in sorted({3, n + 1}):
        paths = _write_all(tmp_path, split_bam(bam, k, "round_robin", block_payload=1700), f"e{k}_")
        one, _ = _qc(paths, tmp_path, f"one_e{k}", *opt, "--vaf-file", str(tmp_path / f"one{k}.vaf"))
        many, _ = _qc(paths, tmp_path, f"many_e{k}", *opt, "--vaf-file", str(tmp_path / f"many{k}.vaf"), "--cuda-devices", devs)
        assert canonical_results(many) == canonical_results(one)
        assert (tmp_path / f"many{k}.vaf").read_bytes() == (tmp_path / f"one{k}.vaf").read_bytes()
