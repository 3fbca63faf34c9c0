"""The CSI restatement (tests/cpp/csi_oracle.c, oracle_build_csi): region queries over its index return exactly the records
that overlap the region, on the micro-BAMs, bamgen shapes 0-4 and hand-built files over references of 2^29 - 1 to 2^31 - 1
bases, at min_shift 12, 14 and 16; no bin's loffset passes a record that overlaps the bin's first window; below 2^29 at
(14, 5) its bins and chunks are the BAI's; and the default depth follows samtools' rule on both sides of every level
threshold."""
import random

import pytest

from baiutil import brute_force, micro_bams, oracle_bai
from csiutil import big_reference_bams, csi_default_depth, csi_region_query, oracle_csi, oracle_csi_keys
from bamutil import write_bam
from helpers import OracleError

MIN_SHIFTS = [12, 14, 16]
_CASES = {}


def case(name):
    """the BAM bytes of a named input"""
    if name not in _CASES:
        if name.startswith("micro:"):
            bam = micro_bams()[name[6:]][0]
        elif name.startswith("shape"):
            from ngs_b200 import ffi
            shape = int(name[5:])
            bam = ffi.synth_bam(shape, {2: 300, 4: 2000}.get(shape, 4000), level=1)[0].tobytes()
        else:
            bam = big_reference_bams()[name]
        _CASES[name] = bam
    return _CASES[name]


NAMES = [f"micro:{n}" for n in sorted(micro_bams())] + [f"shape{s}" for s in range(5)] + sorted(big_reference_bams())


def regions(keys, n_ref, min_shift, depth, seed=1):
    """Per reference: regions that straddle 2^29, 2^30 and the bin boundaries of every level near the records, and random
    ones."""
    rng = random.Random(seed)
    out = []
    for ref in range(n_ref):
        pos = [k[3] for k in keys if k[5] and k[0] == ref]
        if not pos:
            continue
        hi = max(k[4] for k in keys if k[5] and k[0] == ref)
        pts = {1 << 29, 1 << 30}
        for p in rng.sample(pos, min(len(pos), 12)):
            for s in range(min_shift, min_shift + 3 * depth + 1, 3):
                pts.add((p >> s) << s)
                pts.add(((p >> s) + 1) << s)
        for b in sorted(pts):
            if b <= hi + 1000:
                out += [(ref, max(0, b - 1), b + 1), (ref, max(0, b - 5000), b), (ref, b, b + 70000)]
        for _ in range(10):
            a = rng.randrange(0, hi + 1)
            out.append((ref, a, a + rng.choice([1, 300, 20000, 1 << 22])))
        out.append((ref, 0, hi + 1))
    return out


@pytest.mark.parametrize("min_shift", MIN_SHIFTS)
@pytest.mark.parametrize("name", NAMES)
def test_csi_queries_equal_brute_force(name, min_shift):
    from ngs_b200.formats import parse_csi
    bam = case(name)
    csi = oracle_csi(bam, min_shift)
    keys, err, depth = oracle_csi_keys(bam, min_shift)
    assert err is None
    idx = parse_csi(csi)
    assert (idx.min_shift, idx.depth, idx.aux) == (min_shift, depth, b"")
    assert idx.n_no_coor == sum(1 for k in keys if not k[5])
    for ref, beg, end in regions(keys, len(idx.refs), min_shift, depth):
        assert csi_region_query(csi, bam, keys, ref, beg, end) == brute_force(keys, ref, beg, end), (ref, beg, end)


@pytest.mark.parametrize("min_shift", MIN_SHIFTS)
@pytest.mark.parametrize("name", NAMES)
def test_loffset_never_passes_a_record_of_the_bins_first_window(name, min_shift):
    from ngs_b200.formats import parse_csi
    bam = case(name)
    idx = parse_csi(oracle_csi(bam, min_shift))
    keys, _, depth = oracle_csi_keys(bam, min_shift)
    for ref, R in enumerate(idx.refs):
        placed = [k for k in keys if k[5] and k[0] == ref]
        for b, loff in R.loffset.items():
            lv, first = 0, 0
            while first + (1 << 3 * lv) <= b:
                first += 1 << 3 * lv
                lv += 1
            bot = (b - first) << 3 * (depth - lv)
            w0, w1 = bot << min_shift, (bot + 1) << min_shift
            over = [k[7] for k in placed if k[3] < w1 and k[4] > w0]
            assert all(loff <= v for v in over), (ref, b)
            assert any(v >= loff for v in [k[7] for k in placed])


@pytest.mark.parametrize("name", [n for n in NAMES if n.startswith(("micro:", "shape")) and n != "shape4"])
def test_below_2_29_the_csi_holds_the_bais_bins_and_chunks(name):
    from ngs_b200.formats import parse_bai, parse_csi
    bam = case(name)
    c, b = parse_csi(oracle_csi(bam, 14, 5)), parse_bai(oracle_bai(bam))
    assert (c.min_shift, c.depth) == (14, 5)
    assert c.n_no_coor == b.n_no_coor and len(c.refs) == len(b.refs)
    for rc, rb in zip(c.refs, b.refs):
        assert list(rc.bins.items()) == list(rb.bins.items())
        assert (rc.ref_beg, rc.ref_end, rc.n_mapped, rc.n_unmapped) == (rb.ref_beg, rb.ref_end, rb.n_mapped, rb.n_unmapped)
        # the loffset of a leaf bin is the BAI's linear-index entry of its window
        for bn, loff in rc.loffset.items():
            if bn >= 4681:
                assert loff == rb.linear[bn - 4681]


@pytest.mark.parametrize("min_shift", MIN_SHIFTS)
def test_default_depth_on_both_sides_of_every_level_threshold(min_shift):
    from ngs_b200.formats import parse_csi
    n = 0
    while (1 << (min_shift + 3 * n)) - 256 < (1 << 31):
        for L, want in (((1 << (min_shift + 3 * n)) - 256, n), ((1 << (min_shift + 3 * n)) - 255, n + 1)):
            if not 0 < L < (1 << 31):
                continue
            assert csi_default_depth(L, min_shift) == want
            bam, _ = write_bam([("a", 100), ("b", L)], [])
            assert parse_csi(oracle_csi(bam, min_shift)).depth == want, (L, min_shift)
        n += 1


def test_limits_are_refused():
    from csiutil import _at
    # a record past 2^(min_shift + 3 depth), and a reference longer than an explicit depth addresses
    bam, _ = write_bam([("a", (1 << 29) - 300)], [_at((1 << 29) - 350, cigar="100M")])
    assert oracle_csi(bam, 14, 0)  # depth 5 holds it up to 2^29
    bam, _ = write_bam([("a", (1 << 29) - 300)], [_at((1 << 29) - 50, cigar="100M")])
    with pytest.raises(OracleError, match="2\\^29"):
        oracle_csi(bam, 14, 0)
    assert oracle_csi(bam, 14, 6)
    bam, _ = write_bam([("a", (1 << 30) + 1)], [])
    with pytest.raises(OracleError, match="longer"):
        oracle_csi(bam, 14, 5)
