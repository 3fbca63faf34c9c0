"""Read groups on the GPU (NGSQ_F_READ_GROUPS, `qc --cuda-by-read-group`, DESIGN.md section 5, "Read groups").

At the ABI: every group's getters equal the oracle's group filter (tests/cpp/oracle_read_groups.c), the groups add up to the
sample, and the sample's integers are those of a run without the flag — on the four bench shapes with K = 1, 7 and 300
declared groups, with waves of a few blocks (records and the open carry straddle waves) and `-n` at wave and group boundaries;
hand-built aux blocks; a malformed aux field in front of RG; a read longer than the quality table; the refusals.  Through the
driver: each per-group JSON equals the oracle's, the sample JSON is byte-identical to a run without the flag, records in any
order, several files, an index built in the same pass, and several devices (skipped on a box with fewer)."""
import json
import os
import subprocess

import numpy as np
import pytest

from helpers import assert_same_ints, canonical_results, engine_ints
from rgutil import adversarial_records, engine_group_ints, oracle_group_ints, sum_groups, write_rg_bam

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "ngs_b200", "ngs-cuda-qc")
GRCH38 = "GRCh38_no_alt_AnalysisSet"
SEED = 5
E_ARG, E_BAD_RECORD, E_NOMEM, E_QUAL_CAP = -1, -6, -10, -13  # include/ngs_cuda.h


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _rg_engine(bam, ids, n_records=0, launch_blocks=0, quality_positions=0, coverage=True):
    from ngs_b200 import ffi
    flags = ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_VERIFY_CRC | ffi.NGSQ_F_READ_GROUPS | (ffi.NGSQ_F_COVERAGE if coverage else 0)
    eng = ffi.Engine(flags=flags, gc_seed=SEED, max_records=n_records, launch_blocks=launch_blocks, quality_positions=quality_positions)

    class Hook:  # set_read_groups between set_references and the first submit
        def __init__(self, e):
            self.e = e

        def __getattr__(self, k):
            return getattr(self.e, k)

        def set_references(self, *a):
            self.e.set_references(*a)
            self.e.set_read_groups(ids)
    out = engine_ints(bam, n_records=n_records, gc_seed=SEED, coverage=coverage, launch_blocks=launch_blocks, engine=Hook(eng))
    return out, eng


_S = {}


def _synth(shape, k):
    from ngs_b200 import ffi
    key = (shape, min(k, 10))
    if key not in _S:
        _S[key] = ffi.synth_bam(shape, {0: 30000, 1: 12000, 2: 400, 3: 30000}[shape], level=1, read_groups=min(k, 10))
    return _S[key]


def _check(bam, ids, n_records=0, launch_blocks=0, sample=None):
    got, eng = _rg_engine(bam, ids, n_records=n_records, launch_blocks=launch_blocks)
    whole, groups = engine_group_ints(eng, len(ids))
    for g, grp in enumerate(groups):
        if len(ids) > 20 and g not in (0, 1, 9, 10, len(ids) - 1, len(ids)):
            assert grp["general"][0] == 0 or g < 10
            continue
        assert_same_ints(grp, oracle_group_ints(bam, ids, g, n_records=n_records, gc_seed=SEED), coverage=False)
    assert_same_ints(sum_groups(groups), whole, coverage=False)
    if sample is not None:
        assert_same_ints(got, sample)
    eng.close()
    return groups


@pytest.mark.parametrize("k", [1, 7, 300])
@pytest.mark.parametrize("shape", [0, 1, 2, 3])
def test_groups_equal_the_oracle_and_add_up_to_the_sample(shape, k):
    bam, _, _ = _synth(shape, k)
    ids = [f"rg{i}" for i in range(k)]
    sample = engine_ints(bam, gc_seed=SEED)  # without the flag
    groups = _check(bam, ids, sample=sample)
    assert all(int(g["general"][0]) > 0 for g in groups[:min(k, 10)])
    assert groups[-1]["general"][0] == 0
    if shape in (0, 3):  # small waves: records and the open carry straddle waves; -n at wave and group boundaries
        _check(bam, ids, launch_blocks=3, sample=engine_ints(bam, gc_seed=SEED, launch_blocks=3))
        for n in (1, 32, 4096, 12345):
            _check(bam, ids, n_records=n, launch_blocks=5, sample=engine_ints(bam, n_records=n, gc_seed=SEED, launch_blocks=5))


def test_hand_built_aux_blocks():
    from bamutil import as_u8
    ids, rs = adversarial_records()
    bam, _ = write_rg_bam([("chr1", 100000)], rs, ids, block_payload=3000)
    b = as_u8(bam)
    for lb in (0, 2):
        groups = _check(b, ids, launch_blocks=lb, sample=engine_ints(b, gc_seed=SEED, launch_blocks=lb))
        assert all(int(g["general"][0]) for g in groups)


@pytest.mark.parametrize("bad", [b"XZZabc", b"XBq\x01\x00\x00\x00a", b"XQ?", b"XiI\x01\x00"])
def test_a_malformed_field_in_front_of_rg_fails_only_with_the_flag(bad):
    from bamutil import as_u8, rec
    from ngs_b200 import ffi
    from rgutil import aux_z
    rs = [rec(name=f"g{i}", ref=0, pos=i, cigar="4M", seq="ACGT", aux=aux_z("RG", "a")) for i in range(50)]
    rs.append(rec(name="b", ref=0, pos=60, cigar="4M", seq="ACGT", aux=bad + (aux_z("RG", "a") if not bad.endswith(b"c") else b"")))
    bam, _ = write_rg_bam([("chr1", 1000)], rs, ["a"])
    b = as_u8(bam)
    with pytest.raises(ffi.NgsqError) as ei:
        _rg_engine(b, ["a"])
    assert ei.value.code == E_BAD_RECORD
    assert engine_ints(b, gc_seed=SEED)["general"][0] == 51


def test_a_read_longer_than_the_quality_table_reruns_with_the_groups():
    from bamutil import as_u8, rec
    from ngs_b200 import ffi
    from rgutil import aux_z
    import random
    rng = random.Random(2)
    n = 131073
    rs = [rec(name=f"s{i}", ref=0, pos=10 + i, cigar="150M", seq="".join(rng.choice("ACGT") for _ in range(150)),
              qual=[rng.randrange(41) for _ in range(150)], aux=aux_z("RG", ["x", "y"][i % 2])) for i in range(40)]
    rs.append(rec(name="long", ref=0, pos=100, cigar=f"{n}M", seq="".join(rng.choice("ACGT") for _ in range(n)),
                  qual=[rng.randrange(41) for _ in range(n)], aux=aux_z("RG", "y")))
    rs.sort(key=lambda r: r[1]["pos"])
    bam, _ = write_rg_bam([("chr1", 1000000)], rs, ["x", "y"])
    b = as_u8(bam)
    with pytest.raises(ffi.NgsqError) as ei:
        _rg_engine(b, ["x", "y"])
    assert ei.value.code == E_QUAL_CAP
    got, eng = _rg_engine(b, ["x", "y"], quality_positions=n + 1)
    whole, groups = engine_group_ints(eng, 2)
    for g in range(3):
        assert_same_ints(groups[g], oracle_group_ints(b, ["x", "y"], g, gc_seed=SEED), coverage=False)
    assert groups[1]["quality"].shape[0] == n and groups[0]["quality"].shape[0] == 150
    eng.close()


def test_refusals():
    from ngs_b200 import ffi
    bam, _, _ = _synth(0, 7)
    with pytest.raises(ffi.NgsqError) as ei:
        ffi.Engine(flags=ffi.NGSQ_F_COVERAGE | ffi.NGSQ_F_READ_GROUPS)
    assert ei.value.code == E_ARG
    plain = ffi.Engine()
    plain.set_references([1000], [0])
    with pytest.raises(ffi.NgsqError):
        plain.set_read_groups(["a"])
    plain.close()
    eng = ffi.Engine(flags=ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_READ_GROUPS)
    with pytest.raises(ffi.NgsqError):  # before ngsq_set_references
        eng.set_read_groups(["a"])
    eng.set_references([248956422] * 3, [1, 1, 1])
    for bad in (["a", ""], ["a", "b", "a"]):
        with pytest.raises(ffi.NgsqError) as ei:
            eng.set_read_groups(bad)
        assert ei.value.code == E_ARG
    with pytest.raises(ffi.NgsqError) as ei:
        eng.set_read_groups([f"g{i}" for i in range(65535)])
    assert ei.value.code == E_ARG
    with pytest.raises(ffi.NgsqError) as ei:
        eng.set_read_groups([f"g{i}" for i in range(65534)])
    assert ei.value.code == E_NOMEM and "65535 groups" in str(ei.value) and "131072 quality rows" in str(ei.value)
    eng.close()
    ids = [f"rg{i}" for i in range(7)]
    got, eng = _rg_engine(bam, ids)
    eng.select_read_group(3)
    with pytest.raises(ffi.NgsqError) as ei:
        eng.coverage_contig(0, 248956422)
    assert ei.value.code == E_ARG
    with pytest.raises(ffi.NgsqError):
        eng.select_read_group(8)
    eng.select_read_group(-1)
    eng.coverage_contig(0, 248956422)
    eng.reset()
    with pytest.raises(ffi.NgsqError):  # select before finish
        eng.select_read_group(0)
    eng.close()


def test_set_after_submit_is_refused():
    from ngs_b200 import ffi, formats
    bam, _, _ = _synth(0, 7)
    eng = ffi.Engine(flags=ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_READ_GROUPS)
    hdr = formats.read_header(eng, bam)
    eng.set_references([l for _, l in hdr.refs], [0] * len(hdr.refs))
    eng.set_read_groups(["rg0"])
    eng.set_range(hdr.first_voffset, 0)
    eng.submit(np.ascontiguousarray(bam[hdr.first_voffset >> 16:]), hdr.first_voffset >> 16)
    with pytest.raises(ffi.NgsqError) as ei:
        eng.set_read_groups(["rg0", "rg1"])
    assert ei.value.code == E_ARG
    eng.finish()
    eng.close()


# ---------------------------------------------------------------- the driver
def _write(path, data):
    with open(path, "wb") as f:
        f.write(bytes(data))
    return str(path)


def _qc(paths, outdir, prefix, *extra):
    also = [a for p in paths[1:] for a in ("--cuda-also", p)]
    r = subprocess.run([DRIVER, "qc", paths[0], GRCH38, "-o", str(outdir), "-p", prefix, "--cuda-gc-seed", str(SEED)] + also + list(extra),
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    return r.stderr


def _group_files(outdir, prefix, ids):
    return [os.path.join(str(outdir), f"{prefix}.read_group.{i}.results.json") for i in ids]


@pytest.mark.parametrize("shape", [0, 3])
def test_driver_writes_the_oracles_json_per_group(tmp_path, shape):
    bam, bai, _ = _synth(shape, 7)
    ids = [f"rg{i}" for i in range(7)]
    s = _write(tmp_path / "s.bam", bam)
    _write(s + ".bai", bai)
    plain = tmp_path / "plain"
    plain.mkdir()
    _qc([s], plain, "s")
    err = _qc([s], tmp_path, "s", "--cuda-by-read-group")
    assert "INFO   [*] 7 read groups" in err and "WARN" not in err
    assert open(tmp_path / "s.results.json", "rb").read() == open(plain / "s.results.json", "rb").read()
    for g, path in enumerate(_group_files(tmp_path, "s", ids)):
        want = str(tmp_path / f"oracle{g}.json")
        oracle_group_ints(bam, ids, g, gc_seed=SEED, json_path=want)
        assert canonical_results(path) == canonical_results(want), ids[g]
        assert json.load(open(path))["coverage"] is None
    assert not os.path.exists(tmp_path / "s.no_read_group.results.json")
    # --only: that section per group
    only = tmp_path / "only"
    only.mkdir()
    _qc([s], only, "s", "--cuda-by-read-group", "--only", "GC Content")
    j = json.load(open(_group_files(only, "s", ids)[2]))
    assert j["gc_content"] == json.load(open(_group_files(tmp_path, "s", ids)[2]))["gc_content"] and j["general"] is None


def test_driver_ungrouped_records_and_empty_groups(tmp_path):
    from bamutil import as_u8
    ids, rs = adversarial_records()
    bam, bai = write_rg_bam([("chr1", 100000)], rs, ids + ["empty/one", "."])
    s = _write(tmp_path / "a.bam", bam)
    _write(s + ".bai", bai)
    err = _qc([s], tmp_path, "a", "--cuda-by-read-group")
    assert "WARN" in err
    all_ids = ids + ["empty/one", "."]
    names = {"rg1": "rg1", "rg10": "rg10", "lane 2/x": "lane%202%2Fx", "r%g": "r%25g", "empty/one": "empty%2Fone", ".": "."}
    for g, i in enumerate(all_ids):
        path = tmp_path / f"a.read_group.{names[i]}.results.json"
        want = str(tmp_path / f"o{g}.json")
        oracle_group_ints(as_u8(bam), all_ids, g, gc_seed=SEED, json_path=want)
        assert canonical_results(str(path)) == canonical_results(want), i
    j = json.load(open(tmp_path / "a.read_group.empty%2Fone.results.json"))
    assert j["general"]["records"]["total"] == 0 and j["general"]["summary"]["duplication_pct"] is None
    want = str(tmp_path / "ou.json")
    oracle_group_ints(as_u8(bam), all_ids, len(all_ids), gc_seed=SEED, json_path=want)
    assert canonical_results(str(tmp_path / "a.no_read_group.results.json")) == canonical_results(want)


def test_driver_any_order_several_files_and_index(tmp_path):
    from orderutil import reorder
    bam, bai, _ = _synth(3, 7)
    ids = [f"rg{i}" for i in range(7)]
    s = _write(tmp_path / "s.bam", bam)
    _write(s + ".bai", bai)
    _qc([s], tmp_path, "s", "--cuda-by-read-group")
    shuffled, _ = reorder(bam.tobytes(), "random", seed=1)
    u = _write(tmp_path / "u.bam", shuffled)
    _qc([u], tmp_path, "u", "--cuda-by-read-group", "--cuda-any-order")
    for a, b in zip(_group_files(tmp_path, "s", ids), _group_files(tmp_path, "u", ids)):  # shape 3: 2x100, no GC window offsets
        assert canonical_results(a) == canonical_results(b)
    # an index built in the same pass is the index built without the flag
    for name, flag in (("i1", []), ("i2", ["--cuda-by-read-group"])):
        p = _write(tmp_path / f"{name}.bam", bam)
        _qc([p], tmp_path, name, "--cuda-build-index", *flag)
    assert open(tmp_path / "i1.bam.bai", "rb").read() == open(tmp_path / "i2.bam.bai", "rb").read()


def test_driver_several_files_one_group_each(tmp_path):
    from bamutil import rec
    from rgutil import aux_z
    import random
    rng = random.Random(9)
    paths = []
    for lane in range(3):
        rs = [rec(name=f"l{lane}_{i}", flag=[0x41, 0x81, 0x400][i % 3], ref=0, pos=5 * i + lane, mapq=30, cigar="100M", next_ref=0,
                  next_pos=50, tlen=[200, 0, 5000][i % 3], seq="".join(rng.choice("ACGT") for _ in range(100)),
                  qual=[rng.randrange(20, 41) for _ in range(100)], aux=aux_z("RG", f"lane{lane}")) for i in range(500 * (lane + 1))]
        bam, _ = write_rg_bam([("chr1", 100000)], rs, [f"lane{lane}"])
        paths.append(_write(tmp_path / f"lane{lane}.bam", bam))
    _qc(paths, tmp_path, "all", "--cuda-by-read-group")
    for lane in range(3):
        _qc([paths[lane]], tmp_path, f"one{lane}", "--cuda-any-order")
        got = json.load(open(tmp_path / f"all.read_group.lane{lane}.results.json"))
        want = json.load(open(tmp_path / f"one{lane}.results.json"))
        for k in ("general", "gc_content", "template_length", "quality_scores"):
            assert got[k] == want[k], (lane, k)


@pytest.mark.parametrize("n_dev", [2, 4])
def test_several_devices_equal_one(tmp_path, n_dev):
    if _n_gpus() < n_dev:
        pytest.skip(f"needs {n_dev} GPUs")
    bam, bai, _ = _synth(0, 7)
    ids = [f"rg{i}" for i in range(7)]
    s = _write(tmp_path / "s.bam", bam)
    _write(s + ".bai", bai)
    _qc([s], tmp_path, "one", "--cuda-by-read-group")
    _qc([s], tmp_path, "many", "--cuda-by-read-group", "--cuda-devices", ",".join(str(d) for d in range(n_dev)))
    for a, b in zip(_group_files(tmp_path, "one", ids), _group_files(tmp_path, "many", ids)):
        assert canonical_results(a) == canonical_results(b)
