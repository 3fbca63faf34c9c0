"""`qc --cuda-by-read-group` on CPU (ngs_b200/host/read_groups.hpp through tests/cpp/host_read_groups.cpp): the @RG IDs of a
header, the refusals with their messages, the union of the IDs of several files (`--cuda-also`), the file-name escaping, the
usage text, and a group's results JSON from the oracle's integers for that group (the test double of the getters,
tests/cpp/fake_engine.cpp), floats included."""
import os
import subprocess

import numpy as np
import pytest

from helpers import canonical_results
from rgutil import oracle_group_ints

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "ngs_b200", "ngs-cuda-qc")
GRCH38 = "GRCh38_no_alt_AnalysisSet"


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("hostrg") / "host_read_groups")
    subprocess.run(["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-o", out, os.path.join(ROOT, "tests", "cpp", "host_read_groups.cpp"),
                    os.path.join(ROOT, "tests", "cpp", "fake_engine.cpp"), "-lz"], check=True)
    return out


def _run(exe, *args, env=None):
    return subprocess.run([exe] + [str(a) for a in args], capture_output=True, text=True, check=True, env=env).stdout


def _hdr(tmp_path, name, text):
    p = tmp_path / name
    p.write_bytes(text.encode())
    return str(p)


def test_ids_in_header_order_from_any_column(exe, tmp_path):
    text = ("@HD\tVN:1.6\n@SQ\tSN:chr1\tLN:10\n@RG\tID:L1\tSM:a\tPL:ILLUMINA\n@RG\tSM:b\tLB:x\tID:L2\n@PG\tID:notagroup\n"
            "@RG\tPU:f.1\tID:L 3/x\r\n@CO\t@RG\tID:comment\n")
    assert _run(exe, "ids", _hdr(tmp_path, "h.sam", text), "h.bam").splitlines() == ["L1", "L2", "L 3/x"]


@pytest.mark.parametrize("text,msg", [
    ("@HD\tVN:1.6\n@SQ\tSN:chr1\tLN:10\n", "--cuda-by-read-group: the header of h.bam has no @RG line"),
    ("@RG\tID:a\n@RG\tSM:x\n", '--cuda-by-read-group: an @RG line of h.bam has no ID: "@RG\tSM:x"'),
    ("@RG\tID:\tSM:x\n", '--cuda-by-read-group: an @RG line of h.bam has no ID: "@RG\tID:\tSM:x"'),
    ("@RG\tID:a\tSM:x\n@RG\tID:b\n@RG\tID:a\tSM:y\n", '--cuda-by-read-group: the read group ID "a" is declared twice in the header of h.bam'),
])
def test_refused_headers(exe, tmp_path, text, msg):
    assert _run(exe, "ids", _hdr(tmp_path, "h.sam", text), "h.bam").strip() == "error: " + msg


@pytest.mark.parametrize("facet", ["Coverage", "coverage", "Edits", "Genomic Features", "genomic features"])
def test_only_a_sample_facet_is_refused(exe, tmp_path, facet):
    out = _run(exe, "only", facet).strip()
    assert out.startswith(f"error: --cuda-by-read-group cannot be combined with --only {facet}:")
    p = str(tmp_path / "absent.bam")  # the driver refuses it before opening the file
    r = subprocess.run([DRIVER, "qc", p, GRCH38, "--cuda-by-read-group", "--only", facet], capture_output=True, text=True)
    assert r.returncode == 1 and r.stderr.startswith(f"Error: --cuda-by-read-group cannot be combined with --only {facet}:"), r.stderr
    for ok in ("General", "Quality Score", "GC Content", "Template Length"):
        assert _run(exe, "only", ok).strip() == "ok"


def test_union_over_several_files(exe, tmp_path):
    a = _hdr(tmp_path, "a.sam", "@RG\tID:L1\n@RG\tID:L2\n")
    b = _hdr(tmp_path, "b.sam", "@RG\tID:L3\n@RG\tID:L1\n")
    c = _hdr(tmp_path, "c.sam", "@RG\tID:L2\n")
    assert _run(exe, "union", a, b, c).splitlines() == ["L1", "L2", "L3"]
    d = _hdr(tmp_path, "d.sam", "@SQ\tSN:chr1\tLN:5\n")
    assert _run(exe, "union", a, d).strip() == f"error: --cuda-by-read-group: the header of {d} has no @RG line"


def test_escaping_is_injective_and_stays_in_the_directory(exe):
    ids = ["L1", "a.b_c-d", "%", "%25", "a/b", "../x", ".", "..", "a b", "x\ty", "\xe9", "\xff\x80", "A%2F", "a%2Fb"]
    raw = [i.encode("latin-1") for i in ids]
    got = _run(exe, "escape", *[r.hex() for r in raw]).splitlines()
    assert got[:8] == ["L1", "a.b_c-d", "%25", "%2525", "a%2Fb", "..%2Fx", ".", ".."]
    assert got[8:] == ["a%20b", "x%09y", "%E9", "%FF%80", "A%252F", "a%252Fb"]
    assert len(set(got)) == len(got)
    assert all("/" not in g and set(g) <= set("ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789._-%") for g in got)


def test_usage_names_the_flag_and_keeps_the_other_lines():
    r = subprocess.run([DRIVER, "qc", "-h"], capture_output=True, text=True)
    lines = r.stderr.splitlines()
    assert r.returncode == 0
    assert lines[0] == "usage: ngs-cuda-qc qc <BAM> <REFERENCE_GENOME> [-n N] [-o DIR] [-p PREFIX] [--only FACET]"
    assert lines[7].startswith("       ngs-cuda-qc qc <BAM> <REFERENCE_GENOME> --cuda-also <BAM>")
    k = lines.index("       ngs-cuda-qc qc <BAM> <REFERENCE_GENOME> --cuda-by-read-group [the options above]")
    assert k == 10 and "read_group.<ID>.results.json" in lines[k + 1] and "no_read_group.results.json" in lines[k + 2]
    assert lines[k + 5].startswith("       ngs-cuda-qc index <BAM>")


def _dump_group_ints(path, o):
    u = lambda a: np.asarray(a, dtype=np.uint64).ravel()  # noqa: E731
    np.concatenate([u(o["general"]), u(o["tlen_hist"]), u([o["tlen_processed"], o["tlen_ignored"]]), u(o["gc_hist"]), u(o["gc_nuc"]),
                    u(o["gc_rec"]), u([o["quality"].shape[0]]), u(o["quality"]), u([0]), u([0])]).tofile(path)


@pytest.mark.parametrize("k", [3, 10])
def test_a_groups_json_is_the_oracles(exe, tmp_path, k):
    from ngs_b200 import ffi
    bam, _, _ = ffi.synth_bam(0, 4000, level=1, read_groups=k)
    ids = [f"rg{i}" for i in range(k)] + ["declared_but_empty"]
    for g in range(len(ids) + 1):
        want = str(tmp_path / f"o{g}.json")
        o = oracle_group_ints(bam, ids, g, gc_seed=3, json_path=want)
        ints = str(tmp_path / f"g{g}.bin")
        _dump_group_ints(ints, o)
        _run(exe, "group", g, tmp_path, f"h{g}", env=dict(os.environ, NGSQ_FAKE_INTS=ints))
        assert canonical_results(str(tmp_path / f"h{g}.results.json")) == canonical_results(want), g


def _without_id(refs, recs):
    """A BAM whose header has the @RG lines "@RG\tID:L1\tSM:s" and "@RG\tSM:y\tSM:s"."""
    import struct
    from unittest import mock
    import bamutil
    plain = bamutil.header_bytes

    def hdr(rs):
        h = plain(rs)
        n = struct.unpack_from("<i", h, 4)[0]
        text = h[8:8 + n] + b"@RG\tID:L1\tSM:s\n@RG\tSM:y\tSM:s\n"
        return b"BAM\x01" + struct.pack("<i", len(text)) + text + h[8 + n:]
    with mock.patch.object(bamutil, "header_bytes", hdr):
        return bamutil.write_bam(refs, recs)[0]


@pytest.mark.parametrize("case", ["no_rg", "no_id", "twice", "also_no_rg"])
def test_the_driver_refuses_a_header_before_any_device_work(tmp_path, case):
    """On a machine without a GPU an engine cannot be created: the @RG checks must come first (no index is read here)."""
    import bamutil
    from rgutil import write_rg_bam
    recs = [bamutil.rec(name="r", ref=0, pos=1, cigar="4M", seq="ACGT")]
    refs = [("chr1", 1000)]
    good, _ = write_rg_bam(refs, recs, ["L1"])
    bad = {"no_rg": lambda: bamutil.write_bam(refs, recs)[0], "also_no_rg": lambda: bamutil.write_bam(refs, recs)[0],
           "no_id": lambda: _without_id(refs, recs),
           "twice": lambda: write_rg_bam(refs, recs, ["L1", "L1"])[0]}[case]()
    g, b = tmp_path / "g.bam", tmp_path / "b.bam"
    g.write_bytes(good)
    b.write_bytes(bad)
    args = [str(g), "--cuda-also", str(b)] if case == "also_no_rg" else [str(b)]
    r = subprocess.run([DRIVER, "qc", *args[:1], GRCH38, *args[1:], "--cuda-by-read-group", "--cuda-any-order", "-o", str(tmp_path)], capture_output=True, text=True)
    want = {"no_rg": f"the header of {b} has no @RG line", "also_no_rg": f"the header of {b} has no @RG line",
            "no_id": f'an @RG line of {b} has no ID: "@RG\tSM:y\tSM:s"', "twice": f'the read group ID "L1" is declared twice in the header of {b}'}[case]
    assert r.returncode == 1 and r.stderr.splitlines()[-1] == "Error: --cuda-by-read-group: " + want, r.stderr
    assert "CUDA" not in r.stderr
