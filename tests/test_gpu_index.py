"""GPU BAI build (NGSQ_F_INDEX, K13): Engine.bai() must be the oracle's index byte for byte — bamgen shapes, every micro-BAM,
every wave size and submit form — must serve as qc's index, must leave the qc integers untouched when it rides along, and
must fail where `ngs index` fails.  The host driver's `index` command writes the same bytes."""
import os
import subprocess

import numpy as np
import pytest

from baiutil import bad_record_bams, micro_bams, oracle_bai, oracle_keys, placed_minus_one_bam, unsorted_bams
from helpers import assert_same_ints, canonical_results, engine_ints, oracle_ints

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "ngs_b200", "ngs-cuda-qc")
MICRO = micro_bams()


def gpu_bai(bam, flags=None, launch_blocks=0, chunk=None, device=False, engine=None):
    from ngs_b200 import ffi, formats
    bam = np.ascontiguousarray(np.frombuffer(bam, dtype=np.uint8) if isinstance(bam, (bytes, bytearray)) else bam)
    if flags is None:
        flags = ffi.NGSQ_F_INDEX | ffi.NGSQ_F_VERIFY_CRC
    eng = engine or ffi.Engine(flags=flags, launch_blocks=launch_blocks)
    hdr = formats.read_header(eng, bam)
    eng.set_references([l for _, l in hdr.refs], [1 if formats.is_primary(n) else 0 for n, _ in hdr.refs])
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
            piece = bam[o:o + chunk]
            _, _, used = ffi.bgzf_walk(piece, o)
            used = used or bam.size - o
            eng.submit(np.ascontiguousarray(bam[o:o + used]), o)
            o += used
        eng.finish()
    return eng.bai(), eng


def _synth(shape, n, level=1):
    from ngs_b200 import ffi
    return ffi.synth_bam(shape, n, level=level)


@pytest.mark.parametrize("level", [1, 6])
@pytest.mark.parametrize("shape,n", [(0, 60000), (1, 60000), (2, 1500), (3, 60000)])
def test_gpu_index_equals_the_oracle_on_bamgen_shapes(shape, n, level):
    bam, _, _ = _synth(shape, n, level)
    got, eng = gpu_bai(bam)
    assert got == oracle_bai(bam)
    assert eng.stats()["records"] == n


@pytest.mark.parametrize("name", sorted(MICRO) + ["placed_minus_one"])
def test_gpu_index_equals_the_oracle_on_the_micro_bams(name):
    bam = placed_minus_one_bam()[0] if name == "placed_minus_one" else MICRO[name][0]
    for lb in (0, 1):
        got, _ = gpu_bai(bam, launch_blocks=lb)
        assert got == oracle_bai(bam), lb


@pytest.mark.parametrize("form", ["lb7", "lb64", "chunk-70k", "chunk-300k", "chunk-2m", "device"])
@pytest.mark.parametrize("shape,n", [(1, 80000), (2, 1200), (3, 80000)])
def test_wave_boundaries_and_submit_forms_do_not_change_the_bytes(shape, n, form):
    bam, _, _ = _synth(shape, n)
    want = oracle_bai(bam)
    kw = {"lb7": dict(launch_blocks=7), "lb64": dict(launch_blocks=64), "chunk-70k": dict(chunk=70000, launch_blocks=5),
          "chunk-300k": dict(chunk=300000, launch_blocks=3), "chunk-2m": dict(chunk=2 << 20), "device": dict(device=True, launch_blocks=9)}[form]
    got, eng = gpu_bai(bam, **kw)
    assert got == want
    if form != "chunk-2m":
        assert eng.stats()["waves"] > 3


def test_the_gpu_index_serves_qc():
    bam, bai, _ = _synth(1, 60000)
    got, _ = gpu_bai(bam)
    gi = np.frombuffer(got, dtype=np.uint8)
    a, b = oracle_ints(bam, gi, gc_seed=3), oracle_ints(bam, bai, gc_seed=3)
    assert_same_ints(a, b)
    assert a["coverage"]


@pytest.mark.parametrize("shape,n", [(1, 60000), (3, 40000)])
def test_index_alongside_qc_changes_no_integer(shape, n):
    from ngs_b200 import ffi
    bam, bai, _ = _synth(shape, n)
    plain = engine_ints(bam, gc_seed=9, launch_blocks=11)
    flags = ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_COVERAGE | ffi.NGSQ_F_VERIFY_CRC | ffi.NGSQ_F_INDEX
    eng = ffi.Engine(flags=flags, gc_seed=9, launch_blocks=11)
    both = engine_ints(bam, gc_seed=9, engine=eng)
    assert_same_ints(both, plain)
    assert_same_ints(both, oracle_ints(bam, bai, gc_seed=9))
    assert eng.bai() == gpu_bai(bam, launch_blocks=11)[0] == oracle_bai(bam)


def test_an_engine_indexes_again_after_reset():
    from ngs_b200 import ffi
    eng = ffi.Engine(flags=ffi.NGSQ_F_INDEX | ffi.NGSQ_F_VERIFY_CRC, launch_blocks=4)
    for shape, n in ((0, 20000), (3, 30000), (0, 20000)):
        bam, _, _ = _synth(shape, n)
        eng.reset()
        assert gpu_bai(bam, engine=eng)[0] == oracle_bai(bam)


@pytest.mark.parametrize("name", sorted(unsorted_bams()))
def test_unsorted_input_fails_with_the_offset(name):
    from ngs_b200 import ffi
    bam, first_bad = unsorted_bams()[name]
    keys, _ = oracle_keys(bam)
    with pytest.raises(ffi.NgsqError, match=f"virtual offset {keys[first_bad][7]} ") as ex:
        gpu_bai(bam)
    assert ex.value.code == -14


@pytest.mark.parametrize("name", sorted(bad_record_bams()))
def test_malformed_records_fail(name):
    from ngs_b200 import ffi
    with pytest.raises(ffi.NgsqError) as ex:
        gpu_bai(bad_record_bams()[name])
    assert ex.value.code == -6


def test_argument_checks():
    from ngs_b200 import ffi
    with pytest.raises(ffi.NgsqError, match="max_records") as ex:
        ffi.Engine(flags=ffi.NGSQ_F_INDEX, max_records=10)
    assert ex.value.code == -1
    eng = ffi.Engine(flags=ffi.NGSQ_F_INDEX)
    with pytest.raises(ffi.NgsqError, match="CSI"):
        eng.set_references([1 << 29], [0])
    eng.set_references([1000], [0])
    with pytest.raises(ffi.NgsqError, match="end_voffset"):
        eng.set_range(1 << 16, 5 << 16)
    with pytest.raises(ffi.NgsqError, match="ngsq_get_bai"):
        eng.bai()  # before finish
    bam, _ = MICRO["block_starts"]
    got, eng = gpu_bai(bam)
    with pytest.raises(ffi.NgsqError, match="ngsq_reduce") as ex:
        eng.reduce(0)
    assert ex.value.code == -1
    plain = ffi.Engine(flags=ffi.NGSQ_F_RECORD_FACETS)
    with pytest.raises(ffi.NgsqError, match="without NGSQ_F_INDEX"):
        plain.bai()


# ---------------------------------------------------------------- host driver
def _run(args):
    return subprocess.run([DRIVER] + args, capture_output=True, text=True)


def test_driver_index_writes_the_oracles_bai_and_refuses_to_overwrite(tmp_path):
    bam, bai, _ = _synth(1, 50000, level=6)
    p = str(tmp_path / "s.bam")
    bam.tofile(p)
    r = _run(["index", p, "--cuda-chunk-mb", "1"])
    assert r.returncode == 0, r.stderr
    got = open(p + ".bai", "rb").read()
    assert got == oracle_bai(bam)
    before = os.stat(p + ".bai")
    r = _run(["index", p])
    assert r.returncode != 0 and "exists" in r.stderr
    assert open(p + ".bai", "rb").read() == got and os.stat(p + ".bai").st_mtime_ns == before.st_mtime_ns
    # qc over the GPU's index gives the results it gives over bamgen's
    q = str(tmp_path / "w.bam")
    bam.tofile(q)
    bai.tofile(q + ".bai")
    assert _run(["qc", p, "GRCh38_no_alt_AnalysisSet", "-o", str(tmp_path), "-p", "gpu", "--cuda-gc-seed", "4"]).returncode == 0
    assert _run(["qc", q, "GRCh38_no_alt_AnalysisSet", "-o", str(tmp_path), "-p", "writer", "--cuda-gc-seed", "4"]).returncode == 0
    assert canonical_results(str(tmp_path / "gpu.results.json")) == canonical_results(str(tmp_path / "writer.results.json"))


def test_driver_index_io_modes_and_progress(tmp_path):
    bam, _, _ = _synth(3, 40000)
    for i, extra in enumerate([[], ["--cuda-buffered-io", "--cuda-no-crc"], ["--cuda-device", "0", "--cuda-chunk-mb", "2"]]):
        p = str(tmp_path / f"s{i}.bam")
        bam.tofile(p)
        r = _run(["index", p] + extra)
        assert r.returncode == 0, r.stderr
        assert open(p + ".bai", "rb").read() == oracle_bai(bam)
    assert "records" in r.stderr.lower()


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


@pytest.mark.skipif(_n_gpus() < 2, reason="needs two GPUs")
def test_driver_qc_on_two_devices_over_the_gpu_index(tmp_path):
    bam, bai, _ = _synth(1, 300000)
    p, q = str(tmp_path / "g.bam"), str(tmp_path / "w.bam")
    bam.tofile(p)
    bam.tofile(q)
    bai.tofile(q + ".bai")
    assert _run(["index", p]).returncode == 0
    for path, prefix in ((p, "gpu"), (q, "writer")):
        r = _run(["qc", path, "GRCh38_no_alt_AnalysisSet", "-o", str(tmp_path), "-p", prefix, "--cuda-devices", "0,1", "--cuda-gc-seed", "2"])
        assert r.returncode == 0, r.stderr
    assert canonical_results(str(tmp_path / "gpu.results.json")) == canonical_results(str(tmp_path / "writer.results.json"))
