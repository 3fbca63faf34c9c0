"""GPU CSI build (NGSQ_F_INDEX | NGSQ_F_INDEX_CSI, K13 CSI): Engine.csi() must be the oracle's payload byte for byte — bamgen
shapes 0-4, every micro-BAM, references of 2^29 - 1 to 2^31 - 1 bases, every wave size and submit form, at the default
binning and at min_shift 12 and 16 — whole or joined from parts (ngsq_join_csi) wherever the file is cut; it must leave the qc
integers untouched, fail where the oracle fails, and refuse bad arguments.  The host driver's `index --csi` writes the
payload BGZF-compressed."""
import gzip
import os
import subprocess

import numpy as np
import pytest

from baiutil import bgzf_offsets, micro_bams, oracle_keys, placed_minus_one_bam, unsorted_bams
from csiutil import _at, big_reference_bams, oracle_csi, oracle_csi_keys
from bamutil import EOF_BLOCK, write_bam
from helpers import assert_same_ints, engine_ints, oracle_ints
from test_gpu_index import gpu_bai
from test_gpu_index_parts import even_cuts, find_from, run_parts

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "ngs_b200", "ngs-cuda-qc")
MICRO = micro_bams()
BIG = big_reference_bams()
SHIFTS = [None, 12, 16]  # None: the default binning (min_shift 14, samtools' depth)


def csi_engine(min_shift=None, part=False, **kw):
    from ngs_b200 import ffi
    flags = kw.pop("flags", (ffi.NGSQ_F_INDEX_PART if part else ffi.NGSQ_F_INDEX) | ffi.NGSQ_F_VERIFY_CRC) | ffi.NGSQ_F_INDEX_CSI
    eng = ffi.Engine(0, flags=flags, **kw)
    if min_shift is not None:
        eng.set_index_binning(min_shift, 0)
    return eng


def gpu_csi(bam, min_shift=None, launch_blocks=0, chunk=None, device=False, engine=None):
    """test_gpu_index.gpu_bai's submit forms on a CSI engine"""
    from ngs_b200 import ffi, formats
    bam = np.ascontiguousarray(np.frombuffer(bam, dtype=np.uint8) if isinstance(bam, (bytes, bytearray)) else bam)
    eng = engine or csi_engine(min_shift, launch_blocks=launch_blocks)
    hdr = formats.read_header(eng, bam)
    eng.set_references([l for _, l in hdr.refs], [0] * len(hdr.refs))
    eng.set_range(hdr.first_voffset, 0)
    if device:
        import torch
        d = torch.empty(bam.size + 512, dtype=torch.uint8, device="cuda")
        d[: bam.size].copy_(torch.from_numpy(bam))
        torch.cuda.synchronize()
        blocks, n, _ = ffi.bgzf_walk(bam, 0)
        eng.submit_device(d.data_ptr(), bam.size, blocks, n)
        eng.finish()
        del d
    elif chunk is None:
        eng.submit(bam, 0)
        eng.finish()
    else:
        o = 0
        while o < bam.size:
            _, _, used = ffi.bgzf_walk(bam[o:o + chunk], o)
            used = used or bam.size - o
            eng.submit(np.ascontiguousarray(bam[o:o + used]), o)
            o += used
        eng.finish()
    return eng.csi(), eng


def want(bam, min_shift):
    return oracle_csi(bam, 14 if min_shift is None else min_shift, 0)


_SYNTH = {}


def _synth(shape, level=1, n=None):
    from ngs_b200 import ffi
    n = n or {2: 1500, 4: 3000}.get(shape, 60000)
    if (shape, level, n) not in _SYNTH:
        _SYNTH[(shape, level, n)] = ffi.synth_bam(shape, n, level=level)[0]
    return _SYNTH[(shape, level, n)]


@pytest.mark.parametrize("min_shift", SHIFTS)
@pytest.mark.parametrize("level", [1, 6])
@pytest.mark.parametrize("shape", [0, 1, 2, 3, 4])
def test_gpu_csi_equals_the_oracle_on_bamgen_shapes(shape, level, min_shift):
    bam = _synth(shape, level)
    got, eng = gpu_csi(bam, min_shift)
    assert got == want(bam, min_shift)
    assert eng.stats()["records"] == len(oracle_csi_keys(bam)[0])


@pytest.mark.parametrize("min_shift", SHIFTS)
@pytest.mark.parametrize("name", sorted(MICRO) + ["placed_minus_one"] + sorted(BIG))
def test_gpu_csi_equals_the_oracle_on_hand_built_bams(name, min_shift):
    bam = placed_minus_one_bam()[0] if name == "placed_minus_one" else (MICRO[name][0] if name in MICRO else BIG[name])
    for lb in (0, 1):
        got, _ = gpu_csi(bam, min_shift, launch_blocks=lb)
        assert got == want(bam, min_shift), lb


@pytest.mark.parametrize("min_shift", SHIFTS)
@pytest.mark.parametrize("form", ["lb7", "lb64", "chunk-70k", "chunk-300k", "chunk-2m", "device"])
@pytest.mark.parametrize("shape,n", [(1, 80000), (2, 1200), (3, 80000)])
def test_wave_boundaries_and_submit_forms_do_not_change_the_csi(shape, n, form, min_shift):
    bam = _synth(shape, 1, n)
    kw = {"lb7": dict(launch_blocks=7), "lb64": dict(launch_blocks=64), "chunk-70k": dict(chunk=70000, launch_blocks=5),
          "chunk-300k": dict(chunk=300000, launch_blocks=3), "chunk-2m": dict(chunk=2 << 20), "device": dict(device=True, launch_blocks=9)}[form]
    got, eng = gpu_csi(bam, min_shift, **kw)
    assert got == want(bam, min_shift)
    if form != "chunk-2m":
        assert eng.stats()["waves"] > 3


def test_csi_alongside_qc_changes_no_integer():
    from ngs_b200 import ffi
    bam = _synth(1)
    _, bai, _ = ffi.synth_bam(1, 60000, level=1)
    plain = engine_ints(bam, gc_seed=9, launch_blocks=11)
    flags = ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_COVERAGE | ffi.NGSQ_F_VERIFY_CRC | ffi.NGSQ_F_INDEX | ffi.NGSQ_F_INDEX_CSI
    eng = ffi.Engine(flags=flags, gc_seed=9, launch_blocks=11)
    both = engine_ints(bam, gc_seed=9, engine=eng)
    assert_same_ints(both, plain)
    assert_same_ints(both, oracle_ints(bam, bai, gc_seed=9))
    assert eng.csi() == want(bam, None)


# ---------------------------------------------------------------- parts
def _finder_engine(bam):
    """test_gpu_index_parts._finder_engine on a CSI part engine: a BAI engine refuses references of 2^29 bases or more"""
    from ngs_b200 import formats
    eng = csi_engine(part=True)
    hdr = formats.read_header(eng, np.frombuffer(bam, dtype=np.uint8) if isinstance(bam, bytes) else bam)
    eng.set_references([l for _, l in hdr.refs], [0] * len(hdr.refs))
    return eng, hdr


def joined_csi(bam, cuts, min_shift=None, **kw):
    from ngs_b200 import ffi
    engines = [csi_engine(min_shift, part=True, launch_blocks=kw.get("launch_blocks", 0)) for _ in range(len(cuts) + 1)]
    return ffi.join_csi(run_parts(bam, cuts, engines=engines, **kw))


@pytest.mark.parametrize("min_shift", SHIFTS)
@pytest.mark.parametrize("k", [2, 3, 5, 8])
@pytest.mark.parametrize("shape", [0, 2, 3, 4])
def test_joined_csi_equals_one_engine_and_the_oracle(shape, k, min_shift):
    bam = _synth(shape, 1, {2: 1500, 4: 3000}.get(shape, 40000))
    eng, _ = _finder_engine(bam)
    cuts, _ = even_cuts(eng, bam, k)
    assert len(cuts) == k - 1
    assert joined_csi(bam, cuts, min_shift, launch_blocks=5) == gpu_csi(bam, min_shift)[0] == want(bam, min_shift)


@pytest.mark.parametrize("name", sorted(MICRO) + sorted(BIG))
def test_hand_built_bams_cut_at_every_block_start(name):
    from ngs_b200 import ffi
    bam = MICRO[name][0] if name in MICRO else BIG[name]
    w = want(bam, None)
    b = np.frombuffer(bam, dtype=np.uint8)
    eng, hdr = _finder_engine(bam)
    cuts = []
    for coff, _, isize in bgzf_offsets(b):
        if coff <= hdr.first_voffset >> 16 or not isize:
            continue
        v, _ = find_from(eng, b, coff)
        if v and v > hdr.first_voffset and v not in cuts:
            cuts.append(v)
    for v in cuts:
        assert joined_csi(bam, [v]) == w, v
    if cuts:
        assert joined_csi(bam, cuts) == w


@pytest.mark.parametrize("name", sorted(unsorted_bams()))
def test_unsorted_input_fails_with_the_offset_whole_at_a_cut_and_inside_a_part(name):
    from ngs_b200 import ffi
    bam, first_bad = unsorted_bams()[name]
    bad = oracle_keys(bam)[0][first_bad][7]
    for run in (lambda: gpu_csi(bam), lambda: joined_csi(bam, [bad]), lambda: joined_csi(bam, [])):
        with pytest.raises(ffi.NgsqError, match=f"virtual offset {bad} ") as ex:
            run()
        assert ex.value.code == -14


def test_a_record_past_the_addressable_end_fails():
    from ngs_b200 import ffi
    bam, _ = write_bam([("a", (1 << 29) - 300)], [_at((1 << 29) - 50, cigar="100M")])
    with pytest.raises(ffi.NgsqError, match="2\\^29") as ex:
        gpu_csi(bam)
    assert ex.value.code == -6
    assert gpu_csi(bam, engine=_binned(14, 6))[0] == oracle_csi(bam, 14, 6)


def _binned(min_shift, depth, **kw):
    eng = csi_engine(**kw)
    eng.set_index_binning(min_shift, depth)
    return eng


def test_argument_errors():
    from ngs_b200 import ffi

    def refused(fn, match):
        with pytest.raises(ffi.NgsqError, match=match) as ex:
            fn()
        assert ex.value.code == -1
    refused(lambda: ffi.Engine(0, flags=ffi.NGSQ_F_INDEX_CSI), "NGSQ_F_INDEX_CSI")
    refused(lambda: ffi.Engine(0, flags=ffi.NGSQ_F_INDEX_CSI | ffi.NGSQ_F_RECORD_FACETS), "NGSQ_F_INDEX_CSI")
    refused(lambda: ffi.Engine(0, flags=ffi.NGSQ_F_INDEX).set_index_binning(14, 0), "NGSQ_F_INDEX_CSI")
    eng = csi_engine()
    for ms, d in ((11, 0), (25, 0), (14, 8)):
        refused(lambda: eng.set_index_binning(ms, d), "outside")
    eng.set_references([1000], [0])
    refused(lambda: eng.set_index_binning(14, 0), "precede ngsq_set_references")
    # a reference longer than an explicit depth addresses; the default depth takes any 32-bit length
    refused(lambda: _binned(14, 5).set_references([(1 << 29) + 1], [0]), "CSI")
    csi_engine().set_references([(1 << 32) - 1], [0])
    # the getters name each other
    bam = MICRO["block_starts"][0]
    _, c = gpu_csi(bam)
    refused(c.bai, "ngsq_get_csi")
    _, b = gpu_bai(bam)
    refused(b.csi, "ngsq_get_bai")
    # joins: another binning, BAI and CSI parts mixed
    cut = [k[7] for k in oracle_keys(bam)[0]][3]
    p12 = run_parts(bam, [cut], engines=[csi_engine(12, part=True), csi_engine(12, part=True)])
    p16 = run_parts(bam, [cut], engines=[csi_engine(16, part=True), csi_engine(16, part=True)])
    refused(lambda: ffi.join_csi([p12[0], p16[1]]), "binning")
    bai_parts = run_parts(bam, [cut])
    refused(lambda: ffi.join_csi([p12[0], bai_parts[1]]), "ngsq_join_bai")
    refused(lambda: ffi.join_bai([bai_parts[0], p12[1]]), "ngsq_join_csi")
    refused(lambda: p12[0].csi(), "ngsq_join_csi")
    assert ffi.join_csi(p12) == oracle_csi(bam, 12, 0)


# ---------------------------------------------------------------- host driver
def _run(args):
    return subprocess.run([DRIVER] + args, capture_output=True, text=True)


@pytest.mark.parametrize("devices", [[], ["--cuda-devices", "0,0,0"]])
def test_driver_index_csi_writes_bgzf_and_refuses_to_overwrite(tmp_path, devices):
    bam = _synth(4, 6)
    p = str(tmp_path / "s.bam")
    bam.tofile(p)
    r = _run(["index", p, "--csi", "--cuda-chunk-mb", "1"] + devices)
    assert r.returncode == 0, r.stderr
    assert not os.path.exists(p + ".bai")
    got = open(p + ".csi", "rb").read()
    assert got.endswith(EOF_BLOCK)
    assert gzip.decompress(got) == want(bam, None)
    assert all(isize <= 0xFF00 for _, _, isize in bgzf_offsets(got))
    before = os.stat(p + ".csi").st_mtime_ns
    r = _run(["index", p, "--csi"] + devices)
    assert r.returncode != 0 and "exists" in r.stderr
    assert os.stat(p + ".csi").st_mtime_ns == before
    # -m
    q = str(tmp_path / "m.bam")
    bam.tofile(q)
    r = _run(["index", q, "--csi", "-m", "16"] + devices)
    assert r.returncode == 0, r.stderr
    assert gzip.decompress(open(q + ".csi", "rb").read()) == want(bam, 16)


def test_driver_index_without_csi_still_refuses_a_long_reference(tmp_path):
    p = str(tmp_path / "b.bam")
    _synth(4, 1).tofile(p)
    r = _run(["index", p])
    assert r.returncode != 0 and "CSI" in r.stderr
    assert not os.path.exists(p + ".bai") and not os.path.exists(p + ".csi")
    r = _run(["index", p, "-m", "14"])
    assert r.returncode != 0 and "--csi" in r.stderr
