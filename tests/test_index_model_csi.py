"""CPU check of the CSI kernel's per-record logic: ngs_b200/csrc/index.cuh (index_record and index_windows at a CSI binning),
compiled for the host by tools/index_model.cpp in --csi mode, must give every record the oracle's CSI key, bin, window range
and virtual offset, and must reject a record past 2^(min_shift + 3 depth) as the oracle does."""
import pytest

from baiutil import micro_bams
from csiutil import _at, big_reference_bams, oracle_csi_keys
from bamutil import write_bam
from test_index_model import model, run_model  # noqa: F401  (the compiled model fixture)


def check(model, tmp_path, bam, min_shift):
    want, err, depth = oracle_csi_keys(bam, min_shift)
    assert err is None, err
    rows, merr = run_model(model, tmp_path, bam, ["--csi", str(min_shift), str(depth)])
    assert merr is None
    assert len(rows) == len(want)
    for got, k in zip(rows, want):
        ref, pos, bin_, beg, end, placed, unmapped, voff = k
        assert got[:8] == (ref, pos, bin_ if placed else 0, beg, end, placed, unmapped, voff)
        if placed:
            assert got[8:] == (beg >> min_shift, (end - 1) >> min_shift)
    return len(rows)


def run_model(model, tmp_path, bam, extra):  # noqa: F811
    import subprocess
    p = tmp_path / "x.bam"
    p.write_bytes(bytes(bam))
    r = subprocess.run([model, str(p)] + extra, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    rows, err = [], None
    for line in r.stdout.splitlines():
        if line.startswith("error"):
            err = int(line.split()[1])
        else:
            rows.append(tuple(int(x) for x in line.split()))
    return rows, err


@pytest.mark.parametrize("min_shift", [12, 14, 16])
@pytest.mark.parametrize("shape,n", [(0, 5000), (2, 300), (3, 5000), (4, 3000)])
def test_csi_model_matches_oracle_on_bamgen_shapes(model, tmp_path, shape, n, min_shift):
    from ngs_b200 import ffi
    bam, _, _ = ffi.synth_bam(shape, n, level=1)
    assert check(model, tmp_path, bam.tobytes(), min_shift) == n


@pytest.mark.parametrize("min_shift", [12, 14, 16])
def test_csi_model_matches_oracle_on_hand_built_bams(model, tmp_path, min_shift):
    for bam, _ in micro_bams().values():
        check(model, tmp_path, bam, min_shift)
    for bam in big_reference_bams().values():
        check(model, tmp_path, bam, min_shift)


def test_csi_model_rejects_a_record_past_the_limit(model, tmp_path):
    bam, _ = write_bam([("a", (1 << 29) - 300)], [_at((1 << 29) - 50, cigar="100M")])
    _, err, depth = oracle_csi_keys(bam, 14)
    assert err and depth == 5
    _, merr = run_model(model, tmp_path, bam, ["--csi", "14", "5"])
    assert merr == 2
