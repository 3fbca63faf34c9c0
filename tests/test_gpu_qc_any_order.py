"""`qc --cuda-any-order` (DESIGN.md section 5, "Records in any order"): U holds the records of a coordinate-sorted file S in
another order (random, by read name, reversed; tests/orderutil.py), with unplaced and placed unmapped records scattered through
it and records straddling BGZF blocks.  The engine's qc pass is order-free, so U gives S's integers, except the GC window
of reads longer than 101 bases: it is keyed by the record's virtual offset (DESIGN.md section 2, SURVEY F5), so for those the
GC histogram and nucleobase counts must equal the oracle's record pass over U itself.

On one device: the driver's JSON (and `--vaf-file`) for U against S's; U cut at finder anchors into plain qc engines with every
reference split, merged with ngsq_split_arrays and a torch sum, against the oracle on S; a decoy anchor at a cut.  On several
devices (skipped when the box has fewer): the driver against its one-device run."""
import os
import subprocess

import numpy as np
import pytest

from baiutil import oracle_bai
from helpers import assert_same_ints, canonical_results, collect, engine_ints, merge_ints, oracle_ints
from orderutil import ORDERS, reorder

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
        bam, bai, info = ffi.synth_bam(shape, 1500 if shape == 2 else 30000, level=1)
        _S[shape] = (bam, bai, info)
    return _S[shape]


_U = {}


def _unsorted(shape, order):
    if (shape, order) not in _U:
        bam = _synth(shape)[0]
        _U[(shape, order)] = reorder(bam, order, seed=11 + shape, block_payload=0x7100, level=1)[0]
    return _U[(shape, order)]


def _write(path, data):
    with open(path, "wb") as f:
        f.write(bytes(data))
    return str(path)


def _qc(path, outdir, prefix, *extra):
    r = subprocess.run([DRIVER, "qc", path, GRCH38, "-o", str(outdir), "-p", prefix, "--cuda-gc-seed", str(GC_SEED)] + list(extra),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return os.path.join(str(outdir), prefix + ".results.json"), r.stderr


def _gc_of_u(got, u, s_bai):
    """The GC window fields of U's results against the oracle's record pass over U, and the GC invariants."""
    o = oracle_ints(u, s_bai, gc_seed=GC_SEED, coverage=False)
    assert got["histogram"]["values"] == [int(x) for x in o["gc_hist"]]
    nb = got["nucleobases"]
    assert [nb["total_gc_count"], nb["total_at_count"], nb["total_other_count"]] == [int(x) for x in o["gc_nuc"]]
    assert sum(got["histogram"]["values"]) == got["records"]["processed"]
    assert sum(nb.values()) == 100 * got["records"]["processed"]


def assert_json_of_u(got_path, want_path, u, s_bai, gc_window):
    got, want = canonical_results(got_path), canonical_results(want_path)
    if gc_window:
        assert got == want
        return
    g, w = got.pop("gc_content"), want.pop("gc_content")
    assert got == want
    assert g["records"] == w["records"]
    _gc_of_u(g, u, s_bai)


# ---------------------------------------------------------------- the driver on one device
@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("shape", [0, 1, 2, 3])
def test_driver_json_of_u_equals_s(tmp_path, shape, order):
    bam, bai, _ = _synth(shape)
    s = _write(tmp_path / "s.bam", bam)
    _write(s + ".bai", bai)
    want, _ = _qc(s, tmp_path, "s")
    u = _unsorted(shape, order)
    p = _write(tmp_path / "u.bam", u)
    got, _ = _qc(p, tmp_path, "u", "--cuda-any-order")
    assert_json_of_u(got, want, u, bai, gc_window=shape not in LONG_SHAPES)
    assert not os.path.exists(p + ".bai") and not os.path.exists(p + ".csi")


def test_driver_ignores_an_existing_index(tmp_path):
    """A stale .bai (S's, whose offsets mean nothing in U) and a corrupt .csi next to U are neither read nor touched."""
    bam, bai, _ = _synth(3)
    u = _unsorted(3, "random")
    p = _write(tmp_path / "u.bam", u)
    clean, _ = _qc(p, tmp_path, "clean", "--cuda-any-order")
    _write(p + ".bai", bai)
    _write(p + ".csi", b"not a csi")
    before = [os.stat(p + x).st_mtime_ns for x in (".bai", ".csi")]
    got, _ = _qc(p, tmp_path, "stale", "--cuda-any-order")
    assert open(got, "rb").read() == open(clean, "rb").read()
    assert [os.stat(p + x).st_mtime_ns for x in (".bai", ".csi")] == before
    assert open(p + ".bai", "rb").read() == bytes(bai)
    # a .bai that does not parse, alone: the run without the flag fails on it, the run with the flag never reads it
    os.remove(p + ".csi")
    _write(p + ".bai", b"BAI\x01" + b"\xff" * 7)
    r = subprocess.run([DRIVER, "qc", p, GRCH38, "-o", str(tmp_path), "-p", "read", "--cuda-gc-seed", str(GC_SEED)], capture_output=True, text=True)
    assert r.returncode != 0 and "BAM index" in r.stderr, r.stderr
    got, _ = _qc(p, tmp_path, "garbage", "--cuda-any-order")
    assert open(got, "rb").read() == open(clean, "rb").read()


def _edits_files(tmp_path, order):
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
    u = reorder(bam, order, seed=3, block_payload=1700)[0]
    return s, _write(tmp_path / "u.bam", u)


@pytest.mark.parametrize("order", ORDERS)
def test_driver_with_edits_vaf_file_and_features(tmp_path, order):
    s, u = _edits_files(tmp_path, order)
    opt = ["-r", str(tmp_path / "ref.fa"), "-f", str(tmp_path / "m.gff")]
    want, _ = _qc(s, tmp_path, "s", *opt, "--vaf-file", str(tmp_path / "s.vaf"))
    got, _ = _qc(u, tmp_path, "u", *opt, "--vaf-file", str(tmp_path / "u.vaf"), "--cuda-any-order")
    assert canonical_results(got) == canonical_results(want)
    doc = canonical_results(got)
    assert doc["edits"]["vaf_histogram"]["values"] and doc["features"]["records"]["processed"] > 0
    vaf = (tmp_path / "u.vaf").read_bytes()
    assert vaf == (tmp_path / "s.vaf").read_bytes() and vaf.count(b"\n") > 1000


# ---------------------------------------------------------------- shard by shard on one device
def _plain_flags(edits=False):
    from ngs_b200 import ffi
    return ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_COVERAGE | ffi.NGSQ_F_VERIFY_CRC | (ffi.NGSQ_F_EDITS if edits else 0)


def run_cut(bam, cuts, engines=None, fasta=None, launch_blocks=5):
    """One plain qc engine per range [first record, cut 1), .., [last cut, EOF) (None: an empty range), every reference
    declared split; returns (engines, lens, enabled) once every engine finished, before the merge."""
    from ngs_b200 import ffi, formats
    b = np.ascontiguousarray(bam)
    engines = list(engines or [])
    while len(engines) < len(cuts) + 1:
        engines.append(ffi.Engine(0, flags=_plain_flags(fasta is not None), gc_seed=GC_SEED, launch_blocks=launch_blocks))
    hdr = formats.read_header(engines[0], b)
    lens = [l for _, l in hdr.refs]
    enabled = [1 if formats.is_primary(n) else 0 for n, _ in hdr.refs]
    live = [hdr.first_voffset] + [c for c in cuts if c is not None]
    blocks, nb, _ = ffi.bgzf_walk(b)
    k = 0
    for i, e in enumerate(engines[:len(cuts) + 1]):
        e.reset()
        e.set_references(lens, enabled)
        for c, (name, _) in enumerate(hdr.refs):
            if fasta and name in fasta:
                e.set_reference_bases(c, fasta[name])
        for c in range(len(lens)):
            e.split_reference(c)
        if i > 0 and cuts[i - 1] is None:
            e.set_range(0, 0)
        else:
            first, end = live[k], live[k + 1] if k + 1 < len(live) else 0
            k += 1
            lo, hi = formats.shard_byte_range(formats.Shard(first, end, []), blocks, nb, b.size)
            e.set_range(first, end)
            e.submit(np.ascontiguousarray(b[lo:hi]), lo)
        e.finish()
    return engines[:len(cuts) + 1], lens, enabled


def merged_ints(engines, lens, enabled, root=0):
    from test_gpu_split import merge_split
    merge_split(engines, list(range(len(lens))), root)
    got = merge_ints([collect(e, lens, enabled) for e in engines])
    got["records"] = sum(e.stats()["records"] for e in engines)
    return got


def assert_ints_of_u(got, want_s, u, s_bai, gc_window):
    assert_same_ints(got, want_s, gc_window=gc_window)
    if not gc_window:
        o = oracle_ints(u, s_bai, gc_seed=GC_SEED, coverage=False)
        np.testing.assert_array_equal(got["gc_hist"], o["gc_hist"])
        np.testing.assert_array_equal(got["gc_nuc"], o["gc_nuc"])


_WANT = {}


def _oracle_s(shape):
    if shape not in _WANT:
        bam, bai, _ = _synth(shape)
        _WANT[shape] = oracle_ints(bam, bai, gc_seed=GC_SEED)
    return _WANT[shape]


@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("shape", [0, 2, 3])
def test_one_engine_over_u_equals_the_oracle_on_s(shape, order):
    _, bai, info = _synth(shape)
    u = _unsorted(shape, order)
    got = engine_ints(u, gc_seed=GC_SEED, launch_blocks=5)
    assert got["stats"]["records"] == info["n_records"]
    assert_ints_of_u(got, _oracle_s(shape), u, bai, gc_window=shape not in LONG_SHAPES)


@pytest.mark.parametrize("k", [2, 3, 5])
@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("shape", [0, 2, 3])
def test_cut_at_finder_anchors_equals_the_oracle_on_s(shape, order, k):
    from test_gpu_index_parts import _finder_engine, even_cuts
    _, bai, info = _synth(shape)
    u = _unsorted(shape, order)
    finder, _ = _finder_engine(u)
    cuts, _ = even_cuts(finder, u, k)
    assert len(cuts) == k - 1
    engines, lens, enabled = run_cut(u, cuts)
    got = merged_ints(engines, lens, enabled, root=k - 1)
    assert got["records"] == info["n_records"]
    assert_ints_of_u(got, _oracle_s(shape), u, bai, gc_window=shape not in LONG_SHAPES)


@pytest.mark.parametrize("order", ORDERS)
def test_edits_cut_at_finder_anchors_equal_one_engine(order):
    """Edits' per-position counters of every contig summed onto the root and its VAF pass run after the merge."""
    from test_gpu_index_parts import _finder_engine, even_cuts
    from test_gpu_split import _edits_case
    refs = (("chr2", 8_000), ("chr1", 70_000), ("chrM", 5_000))
    bam, _, fasta, _ = _edits_case(refs, seed=29)
    u = reorder(bam, order, seed=5, block_payload=2900)[0]
    from test_gpu_split import merge_split
    whole, _, _ = run_cut(bam, [], fasta=fasta)
    merge_split(whole, list(range(len(refs))), 0)  # one engine with every reference declared split resolves them itself
    one, two, vaf, n = whole[0].edits()
    want = [whole[0].edit_positions(c, L) for c, (_, L) in enumerate(refs)]
    assert vaf.sum() > 0
    finder, _ = _finder_engine(u)
    cuts, _ = even_cuts(finder, u, 4)
    engines, lens, enabled = run_cut(u, cuts, fasta=fasta)
    merge_split(engines, list(range(len(refs))), 1)
    got = [e.edits() for e in engines]
    np.testing.assert_array_equal(sum(g[0] for g in got), one)
    np.testing.assert_array_equal(sum(g[1] for g in got), two)
    np.testing.assert_array_equal(sum(g[2] for g in got), vaf)
    assert sum(g[3] for g in got) == n
    for c, (_, L) in enumerate(refs):
        pos = [e.edit_positions(c, L) for e in engines]
        np.testing.assert_array_equal(pos[1][0], want[c][0])
        np.testing.assert_array_equal(pos[1][1], want[c][1])
        assert all(not p[0].any() and not p[1].any() for i, p in enumerate(pos) if i != 1)


def test_a_decoy_anchor_is_refuted_and_the_rerun_gives_the_same_integers():
    """The driver's recovery (run_parts) on plain qc engines: the part in front of a false anchor fails with NGSQ_E_CHAIN or
    NGSQ_E_TRUNCATED, the cut is dropped, that part runs again over both ranges and the next engine over an empty one."""
    from ngs_b200 import ffi
    from test_gpu_index_parts import _finder_engine, decoy_case, find_from
    from baiutil import bgzf_offsets
    bam, _ = decoy_case()
    want = oracle_ints(bam, np.frombuffer(oracle_bai(bam), dtype=np.uint8), gc_seed=GC_SEED)
    decoy_block = [c for c, _, isize in bgzf_offsets(bam) if isize][2]
    finder, _ = _finder_engine(bam)
    v, _ = find_from(finder, bam, decoy_block)
    assert v == decoy_block << 16
    engines = [ffi.Engine(0, flags=_plain_flags(), gc_seed=GC_SEED, launch_blocks=5) for _ in range(2)]
    with pytest.raises(ffi.NgsqError) as ex:
        run_cut(bam, [v], engines=engines)
    assert ex.value.code in (-8, -3)
    engines, lens, enabled = run_cut(bam, [None], engines=engines)
    got = merged_ints(engines, lens, enabled, root=1)
    assert got["records"] == want["pass1_records"]
    assert_same_ints(got, want)


# ---------------------------------------------------------------- several devices
@pytest.mark.parametrize("n", [2, 4])
def test_driver_on_several_devices_equals_one(tmp_path, n):
    if _n_gpus() < n:
        pytest.skip(f"needs {n} GPUs")
    devs = ",".join(str(i) for i in range(n))
    for shape in (1, 2):
        u = _write(tmp_path / f"u{shape}.bam", _unsorted(shape, "random"))
        one, _ = _qc(u, tmp_path, f"one{shape}", "--cuda-any-order")
        many, err = _qc(u, tmp_path, f"many{shape}", "--cuda-any-order", "--cuda-devices", devs)
        assert "every reference split" in err
        assert canonical_results(many) == canonical_results(one)
    s, u = _edits_files(tmp_path, "queryname")
    opt = ["-r", str(tmp_path / "ref.fa"), "-f", str(tmp_path / "m.gff"), "--cuda-any-order"]
    one, _ = _qc(u, tmp_path, "one_e", *opt, "--vaf-file", str(tmp_path / "one.vaf"))
    many, _ = _qc(u, tmp_path, "many_e", *opt, "--vaf-file", str(tmp_path / "many.vaf"), "--cuda-devices", devs)
    assert canonical_results(many) == canonical_results(one)
    assert (tmp_path / "many.vaf").read_bytes() == (tmp_path / "one.vaf").read_bytes()


def test_driver_on_two_devices_recovers_from_a_decoy(tmp_path):
    if _n_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    from test_gpu_index_parts import decoy_case
    bam, _ = decoy_case()
    p = _write(tmp_path / "d.bam", bam)
    one, _ = _qc(p, tmp_path, "one", "--cuda-any-order")
    two, err = _qc(p, tmp_path, "two", "--cuda-any-order", "--cuda-devices", "0,1")
    assert "not a record start" in err
    assert canonical_results(two) == canonical_results(one)
