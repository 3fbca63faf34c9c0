"""The BAI oracle (tests/cpp/bai_oracle.c: oracle_build_bai, the index contract of DESIGN.md section 4 K13)
against the two in-repo BAI writers — tests/bamutil.py byte for byte on micro-BAMs, tools/bamgen.cpp up to its clamped
linear index — and against a convention-free check: a standard region query over the oracle's index returns exactly the
records that overlap the region."""
import pytest

from baiutil import (REFS, bad_record_bams, brute_force, micro_bams, oracle_bai, oracle_keys, placed_minus_one_bam, region_query,
                     unsorted_bams)
from helpers import OracleError

MICRO = micro_bams()


@pytest.mark.parametrize("name", sorted(MICRO))
def test_oracle_equals_the_python_writer_byte_for_byte(name):
    bam, want = MICRO[name]
    assert oracle_bai(bam) == want


def test_a_placed_record_without_a_position_is_in_no_bin():
    bam, want = placed_minus_one_bam()
    assert oracle_bai(bam) == want


def test_micro_bams_meet_the_rules_they_are_named_for():
    from ngs_b200.formats import parse_bai
    bai = {k: parse_bai(oracle_bai(v[0])) for k, v in MICRO.items()}
    assert 0 in bai["bin0"].refs[0].bins
    assert bai["overhang"].refs[3].linear and len(bai["overhang"].refs[3].linear) == 4 > (16390 >> 14) + 1
    assert bai["empty_middle"].refs[1].bins == {} and bai["empty_middle"].refs[2].bins and bai["empty_middle"].n_no_coor == 3
    assert bai["unplaced_tail"].n_no_coor == 4 and all(not r.bins for r in bai["unplaced_tail"].refs)
    assert bai["header_only"].n_no_coor == 0 and all(not r.bins and not r.linear for r in bai["header_only"].refs)
    z = bai["zero_span_unmapped"].refs[0]
    assert z.n_unmapped == 6 and z.n_mapped == 6 and len(z.linear) == 6
    keys, _ = oracle_keys(MICRO["block_starts"][0])
    assert sum(1 for k in keys if k[7] & 0xFFFF == 0) >= 3  # records at offset 0 of their block
    keys, _ = oracle_keys(MICRO["spanning"][0])
    assert len({k[7] >> 16 for k in keys}) == len(keys)  # every record starts in a block of its own


@pytest.mark.parametrize("shape,n", [(0, 30000), (1, 30000), (2, 1500), (3, 30000)])
def test_oracle_equals_bamgen_except_its_clamped_linear_index(shape, n):
    from ngs_b200 import ffi
    from ngs_b200.formats import parse_bai, parse_bam_header
    import gzip
    bam, bai, _ = ffi.synth_bam(shape, n, level=1)
    got, want = parse_bai(oracle_bai(bam)), parse_bai(bai.tobytes())
    _, refs, _ = parse_bam_header(gzip.decompress(bam.tobytes()))
    assert got.n_no_coor == want.n_no_coor and len(got.refs) == len(want.refs)
    for (name, L), g, w in zip(refs, got.refs, want.refs):
        assert list(g.bins.items()) == list(w.bins.items()), name  # bins in order of first use, chunks in file order
        assert (g.ref_beg, g.ref_end, g.n_mapped, g.n_unmapped) == (w.ref_beg, w.ref_end, w.n_mapped, w.n_unmapped), name
        # bamgen clamps windows to L >> 14; the oracle grows the array for reads that overhang the contig end
        assert len(w.linear) == min(len(g.linear), (L >> 14) + 1), name
        assert g.linear[: len(w.linear)] == w.linear, name
    assert sum(len(r.bins) for r in got.refs) > 3


@pytest.mark.parametrize("source", ["micro", "shape0", "shape3"])
def test_region_queries_over_the_oracle_index_return_exactly_the_overlapping_records(source):
    from ngs_b200 import ffi
    if source == "micro":
        cases = [(v[0], REFS) for v in MICRO.values()]
    else:
        import gzip
        from ngs_b200.formats import parse_bam_header
        bam, _, _ = ffi.synth_bam(int(source[-1]), 20000, level=1)
        cases = [(bam.tobytes(), parse_bam_header(gzip.decompress(bam.tobytes()))[1])]
    checked = 0
    for bam, refs in cases:
        bai = oracle_bai(bam)
        keys, err = oracle_keys(bam)
        assert err is None
        for ref, (_, L) in enumerate(refs):
            span = min(L, 1 << 26) + 50000
            for beg in sorted({0, 1, 16383, 16384, span // 7, span // 3, span // 2, span - 100, (1 << 26) - 10}):
                for width in (1, 100, 20000, 1 << 20):
                    want = brute_force(keys, ref, beg, beg + width)
                    assert region_query(bai, bam, keys, ref, beg, beg + width) == want, (ref, beg, width)
                    checked += len(want)
    assert checked > 0


@pytest.mark.parametrize("name", sorted(unsorted_bams()))
def test_unsorted_input_is_refused(name):
    bam, first_bad = unsorted_bams()[name]
    keys, _ = oracle_keys(bam)
    with pytest.raises(OracleError, match=f"unsorted records: the record at virtual offset {keys[first_bad][7]} "):
        oracle_bai(bam)


@pytest.mark.parametrize("name", sorted(bad_record_bams()))
def test_malformed_records_are_refused(name):
    bam = bad_record_bams()[name]
    with pytest.raises(OracleError):
        oracle_bai(bam)
    _, err = oracle_keys(bam)
    assert err

