"""CPU check of the BAI kernel's per-record logic: ngs_b200/csrc/index.cuh (index_record, index_windows), compiled for the
host by tools/index_model.cpp, must give every record of bamgen's shapes and of the micro-BAMs the oracle's key, bin,
window range and virtual offset, and must reject the records the oracle rejects."""
import os
import subprocess

import pytest

from baiutil import bad_record_bams, micro_bams, oracle_keys, placed_minus_one_bam

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def model(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("index") / "index_model")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tools", "index_model.cpp"), "-lz"], check=True)
    return exe


def run_model(model, tmp_path, bam):
    p = tmp_path / "x.bam"
    p.write_bytes(bytes(bam))
    r = subprocess.run([model, str(p)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    rows, err = [], None
    for line in r.stdout.splitlines():
        if line.startswith("error"):
            err = int(line.split()[1])
        else:
            rows.append(tuple(int(x) for x in line.split()))
    return rows, err


def check(model, tmp_path, bam):
    want, err = oracle_keys(bam)
    assert err is None, err
    rows, merr = run_model(model, tmp_path, bam)
    assert merr is None
    assert len(rows) == len(want)
    for got, k in zip(rows, want):
        ref, pos, bin_, beg, end, placed, unmapped, voff = k
        assert got[:8] == (ref, pos, bin_ if placed else 0, beg, end, placed, unmapped, voff)
        if placed:
            assert got[8:] == (beg >> 14, (end - 1) >> 14)
    return len(rows)


@pytest.mark.parametrize("shape,n", [(0, 20000), (1, 20000), (2, 1000), (3, 20000)])
def test_model_matches_oracle_on_bamgen_shapes(model, tmp_path, shape, n):
    from ngs_b200 import ffi
    bam, _, _ = ffi.synth_bam(shape, n, level=1)
    assert check(model, tmp_path, bam.tobytes()) == n


def test_model_matches_oracle_on_the_micro_bams(model, tmp_path):
    for name, (bam, _) in micro_bams().items():
        check(model, tmp_path, bam)
    check(model, tmp_path, placed_minus_one_bam()[0])


@pytest.mark.parametrize("name", sorted(bad_record_bams()))
def test_model_rejects_what_the_oracle_rejects(model, tmp_path, name):
    bam = bad_record_bams()[name]
    want, err = oracle_keys(bam)
    assert err and not want
    _, merr = run_model(model, tmp_path, bam)
    assert merr == (2 if name == "too_long" else 1)
