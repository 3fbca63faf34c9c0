"""`qc --cuda-any-order` on CPU: the flags it cannot be combined with are refused before the BAM is opened, and the plan for
records in any order (ngs_b200/host/bam.hpp: plan_shards_any_order, through tests/cpp/host_any_order.cpp with a record finder
backed by the truth) cuts an unsorted file into contiguous shards that partition its records, with every reference split."""
import os
import subprocess

import pytest

from orderutil import ORDERS, reorder
from test_host_unindexed_cpu import walk

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "ngs_b200", "ngs-cuda-qc")
GRCH38 = "GRCh38_no_alt_AnalysisSet"


def _run(args):
    return subprocess.run([DRIVER] + args, capture_output=True, text=True)


@pytest.mark.parametrize("extra,named", [(["-n", "10"], "-n"), (["--num-records", "10"], "-n"),
                                         (["--cuda-build-index"], "--cuda-build-index"),
                                         (["--cuda-build-index", "--cuda-csi"], "--cuda-build-index"),
                                         (["--cuda-csi"], "--cuda-csi")])
def test_conflicting_flags_are_refused(tmp_path, extra, named):
    p = str(tmp_path / "absent.bam")  # refused before the file is opened
    for args in (["qc", p, GRCH38, "--cuda-any-order"] + extra, ["qc", p, GRCH38] + extra + ["--cuda-any-order"]):
        r = _run(args)
        assert r.returncode == 1, r.stderr
        assert r.stderr.startswith(f"Error: --cuda-any-order cannot be combined with {named}:"), r.stderr
        assert "absent.bam" not in r.stderr and not os.path.exists(p + ".bai")


def test_usage_names_the_flag():
    r = _run(["qc", "-h"])
    assert r.returncode == 0 and "--cuda-any-order" in r.stderr


def test_the_missing_index_error_is_unchanged_without_the_flag(tmp_path):
    from ngs_b200 import ffi
    bam, _, _ = ffi.synth_bam(0, 2000, level=1)
    p = str(tmp_path / "x.bam")
    bam.tofile(p)
    out = ["-o", str(tmp_path), "-p", "x"]
    r = _run(["qc", p, GRCH38] + out)
    assert r.returncode == 1
    assert r.stderr.splitlines()[-1] == f"Error: Could not find BAM index at {p}.bai. Please index the BAM first (`ngs index`)."
    # with the flag no index is asked for: the run goes on to the engine (and succeeds where there is a GPU)
    r = _run(["qc", p, GRCH38, "--cuda-any-order"] + out)
    assert "Could not find BAM index" not in r.stderr
    assert r.returncode == 0 or "CUDA engine" in r.stderr, r.stderr


@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("anyorder") / "host_any_order")
    subprocess.run(["g++", "-O1", "-std=c++17", "-o", out, os.path.join(ROOT, "tests", "cpp", "host_any_order.cpp"),
                    "-L" + os.path.join(ROOT, "ngs_b200"), "-lngs_cuda", "-Wl,-rpath," + os.path.join(ROOT, "ngs_b200")], check=True)
    return out


_FILES = {}


def _unsorted(shape, order):
    from ngs_b200 import ffi, formats
    if (shape, order) not in _FILES:
        bam, _, _ = ffi.synth_bam(shape, 1500 if shape == 2 else 20000, level=1)
        u, _ = reorder(bam, order, seed=shape, block_payload=0x9000, level=1)
        raw = bytes(u)
        n_ref = len(formats.parse_bam_header(_header(raw))[1])
        _FILES[(shape, order)] = (raw, n_ref)
    return _FILES[(shape, order)]


def _header(raw):
    import zlib
    bsize = int.from_bytes(raw[16:18], "little") + 1
    return zlib.decompress(raw[18:bsize - 8], -15)  # the header has a block of its own (orderutil.reorder)


@pytest.mark.parametrize("n", [1, 2, 3, 5, 8])
@pytest.mark.parametrize("order", ORDERS)
@pytest.mark.parametrize("shape", [0, 1, 2, 3])
def test_the_plan_partitions_the_records_and_splits_every_reference(exe, tmp_path, shape, order, n):
    raw, n_ref = _unsorted(shape, order)
    blocks, first, recs = walk(raw)
    p, t = tmp_path / "u.bam", tmp_path / "truth.txt"
    p.write_bytes(raw)
    t.write_text("".join(f"{v} {r}\n" for v, r in recs))
    out = subprocess.run([exe, str(p), str(first), str(n_ref), str(n), str(t)], capture_output=True, text=True, check=True).stdout
    assert not out.startswith("error"), out
    lines = out.splitlines()
    rows = [[int(x) for x in ln.split()] for ln in lines[:n]]
    split = [int(x) for x in lines[n].split()[1:]]
    dropped = int(lines[n + 1].split()[1])
    assert len(rows) == n
    live = [r for r in rows if not r[2]]
    if n == 1:
        assert rows == [[first, 0, 0]] and split == [] and dropped == 0  # one shard, nothing to merge
        return
    assert split == list(range(n_ref))
    assert dropped == n - len(live) and all(r[2] for r in rows[len(live):])
    assert live[0][0] == first and live[-1][1] == 0
    assert all(a[1] == b[0] and a[0] < b[0] for a, b in zip(live, live[1:]))  # contiguous, in file order
    starts = {v for v, _ in recs}
    assert all(r[0] in starts for r in live[1:])  # every cut is a record start
    # each record in exactly one shard
    bounds = [r[0] for r in live] + [1 << 64]
    owners = [sum(1 for a, b in zip(bounds, bounds[1:]) if a <= v < b) for v, _ in recs]
    assert owners == [1] * len(recs)
    if order == "random" and len(live) > 1:
        # the anchors' references alone would miss contigs with records on both sides of a cut
        anchor_refs = {r for v, r in recs if v in set(x[0] for x in live[1:])}
        cut = live[1][0]
        both = {r for v, r in recs if v < cut and r >= 0} & {r for v, r in recs if v >= cut and r >= 0}
        assert both - anchor_refs
