"""Read groups on CPU: the oracle's group filter (tests/cpp/oracle_read_groups.c) against an independent Python restatement of
htslib's bam_aux_get rule, group by group, on generator BAMs with K read groups and on hand-built aux blocks; the groups and
the ungrouped records add up to the whole file; and the generator with K = 1 writes the bytes it wrote without the option."""
import hashlib

import numpy as np
import pytest

from helpers import OracleError, assert_same_ints, oracle_ints
from rgutil import adversarial_records, oracle_group_ints, python_group_ints, record_group, sum_groups, write_rg_bam


def _check_groups(bam, ids, seed):
    whole = oracle_group_ints(bam, ids, -1, gc_seed=seed)
    groups = []
    for g in range(len(ids) + 1):
        want = oracle_group_ints(bam, ids, g, gc_seed=seed)
        assert_same_ints(python_group_ints(bam.tobytes(), ids, g, gc_seed=seed), want, coverage=False)
        groups.append(want)
    assert_same_ints(sum_groups(groups), whole, coverage=False)
    return groups


@pytest.mark.parametrize("k", [1, 3, 10])
def test_oracle_and_python_agree_per_group_on_generator_bams(k):
    from ngs_b200 import ffi
    bam, bai, _ = ffi.synth_bam(0, 3000, level=1, read_groups=k)
    ids = [f"rg{i}" for i in range(k)]
    groups = _check_groups(bam, ids, seed=7)
    assert groups[-1]["general"][0] == 0  # every generator record carries a declared group
    assert all(g["general"][0] > 0 for g in groups[:-1])
    # the unfiltered run of the group oracle is the oracle's own pass 1
    o = oracle_ints(bam, bai, gc_seed=7, coverage=False)
    assert_same_ints(oracle_group_ints(bam, ids, -1, gc_seed=7), o, coverage=False)


def test_oracle_and_python_agree_on_hand_built_aux_blocks():
    from bamutil import as_u8
    ids, rs = adversarial_records()
    bam, _ = write_rg_bam([("chr1", 100000)], rs, ids, block_payload=3000)
    b = as_u8(bam)
    groups = _check_groups(b, ids, seed=3)
    n = [int(g["general"][0]) for g in groups]
    assert all(n), n  # every declared ID and the ungrouped records occur
    # rg1 / rg10 are told apart; the first of two RG tags decides
    assert record_group(rs[0][0][4:], ids) == 0 and record_group(rs[3][0][4:], ids) == 1 and record_group(rs[8 * 3][0][4:], ids) == 1


@pytest.mark.parametrize("bad", [b"XZZabc", b"XBq\x01\x00\x00\x00a", b"XQ?", b"XiI\x01\x00", b"XB"])
def test_a_malformed_field_in_front_of_rg_fails(bad):
    from bamutil import as_u8, rec
    from rgutil import aux_z
    good = rec(name="g", ref=0, pos=1, cigar="4M", seq="ACGT", aux=aux_z("RG", "a"))
    broken = rec(name="b", ref=0, pos=2, cigar="4M", seq="ACGT", aux=bad + (aux_z("RG", "a") if bad[-1:] != b"c" else b""))
    bam, _ = write_rg_bam([("chr1", 1000)], [good, broken], ["a"])
    with pytest.raises(OracleError):
        oracle_group_ints(as_u8(bam), ["a"], 0)
    with pytest.raises(ValueError):
        record_group(broken[0][4:], ["a"])
    # behind the RG field nothing is read
    after = rec(name="c", ref=0, pos=3, cigar="4M", seq="ACGT", aux=aux_z("RG", "a") + b"XQ?")
    bam, _ = write_rg_bam([("chr1", 1000)], [good, after], ["a"])
    assert oracle_group_ints(as_u8(bam), ["a"], 0)["general"][0] == 2


def test_n_counts_every_record():
    from ngs_b200 import ffi
    bam, _, _ = ffi.synth_bam(0, 2000, level=1, read_groups=3)
    ids = ["rg0", "rg1", "rg2"]
    for n in (1, 31, 32, 33, 1000):
        per = [int(oracle_group_ints(bam, ids, g, n_records=n)["general"][0]) for g in range(4)]
        assert sum(per) == n


def test_generator_with_one_read_group_writes_the_golden_bytes():
    from ngs_b200 import ffi
    import ctypes as C
    ffi._load_synth()  # test_golden.py pins synth_bam's bytes; K = 1 must reproduce them
    for shape in (0, 1, 2, 3):  # the bench shapes: synth_bam_rg(K = 1) is synth_bam
        a, _, _ = ffi.synth_bam(shape, 3000, level=1)
        b, bi, info = C.c_void_p(), C.c_void_p(), ffi.SynthInfo()
        assert ffi._synth.synth_bam_rg(shape, 3000, 0x5EED0001 + shape, 1, 0, 1, C.byref(b), C.byref(bi), C.byref(info)) == 0
        got = np.ctypeslib.as_array(C.cast(b, C.POINTER(C.c_uint8)), shape=(info.bam_bytes,)).copy()
        ffi._synth.synth_free(b)
        ffi._synth.synth_free(bi)
        assert hashlib.sha256(got.tobytes()).hexdigest() == hashlib.sha256(a.tobytes()).hexdigest()
    # K > 1 keeps every record's length: the inflated size grows by the header's extra @RG lines only
    one, _, i1 = ffi.synth_bam(0, 3000, level=1)
    ten, _, i10 = ffi.synth_bam(0, 3000, level=1, read_groups=10)
    assert i10["inflated_bytes"] - i1["inflated_bytes"] == sum(len(f"@RG\tID:rg{k}\tSM:synthetic\n") for k in range(1, 10))
