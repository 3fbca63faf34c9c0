"""`qc --cuda-also` on CPU: the flags it cannot be combined with and unusable files are refused before any device work; files
whose reference sequences differ are named with the first reference that differs (bam.hpp: check_same_dictionary); and the plan
for several files (bam.hpp: assign_files, devices_per_file, plan_files, through tests/cpp/host_multi_file.cpp with a record
finder backed by the truth) queues whole files largest-first, or cuts each file between its devices."""
import os
import subprocess

import pytest

from splitutil import SPLITS, split_bam
from test_host_unindexed_cpu import walk

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "ngs_b200", "ngs-cuda-qc")
GRCH38 = "GRCh38_no_alt_AnalysisSet"


def _run(args):
    return subprocess.run([DRIVER] + args, capture_output=True, text=True)


@pytest.mark.parametrize("extra,named", [(["-n", "10"], "-n"), (["--num-records", "10"], "-n"),
                                         (["--cuda-build-index"], "--cuda-build-index"),
                                         (["--cuda-build-index", "--cuda-csi"], "--cuda-build-index"),
                                         (["--cuda-csi"], "--cuda-csi"),
                                         (["--cuda-any-order", "-n", "3"], "-n")])
def test_conflicting_flags_are_refused(tmp_path, extra, named):
    p, q = str(tmp_path / "absent.bam"), str(tmp_path / "other.bam")  # refused before either file is opened
    for args in (["qc", p, GRCH38, "--cuda-also", q] + extra, ["qc", p, GRCH38] + extra + ["--cuda-also", q]):
        r = _run(args)
        assert r.returncode == 1, r.stderr
        assert r.stderr.startswith(f"Error: --cuda-also cannot be combined with {named}:"), r.stderr
        assert "absent.bam" not in r.stderr and not os.path.exists(p + ".bai")


def _bam(tmp_path, name="s.bam"):
    from ngs_b200 import ffi
    bam, _, _ = ffi.synth_bam(3, 2000, level=1)
    p = str(tmp_path / name)
    bam.tofile(p)
    return p


def test_a_missing_file_is_refused(tmp_path):
    p = _bam(tmp_path)
    missing = str(tmp_path / "missing.bam")
    r = _run(["qc", p, GRCH38, "--cuda-also", p, "--cuda-also", missing, "-o", str(tmp_path)])
    assert r.returncode == 1
    assert r.stderr.splitlines()[-1] == f"Error: cannot open {missing}"
    assert not os.path.exists(tmp_path / "s.bam.results.json")


@pytest.mark.parametrize("name", ["reads.sam", "reads.cram", "reads", "reads.bam.bai"])
def test_a_file_not_named_bam_is_refused(tmp_path, name):
    p = _bam(tmp_path)
    other = tmp_path / name
    other.write_bytes(open(p, "rb").read())
    r = _run(["qc", p, GRCH38, "--cuda-also", str(other), "-o", str(tmp_path)])
    assert r.returncode == 1
    assert r.stderr.splitlines()[-1] == f"Error: could not open {other}: expected a .bam file"


def test_usage_names_the_flag_and_keeps_the_one_file_text():
    r = _run(["qc", "-h"])
    assert r.returncode == 0
    lines = r.stderr.splitlines()
    assert lines[0] == "usage: ngs-cuda-qc qc <BAM> <REFERENCE_GENOME> [-n N] [-o DIR] [-p PREFIX] [--only FACET]"
    assert lines[6] == "                  with -n, --cuda-build-index or --cuda-csi)"
    assert lines[7].startswith("       ngs-cuda-qc qc <BAM> <REFERENCE_GENOME> --cuda-also <BAM>")
    assert any(ln.startswith("       ngs-cuda-qc index <BAM>") for ln in lines[8:])


# ---------------------------------------------------------------- the harness
@pytest.fixture(scope="module")
def exe(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("multifile") / "host_multi_file")
    subprocess.run(["g++", "-O1", "-std=c++17", "-o", out, os.path.join(ROOT, "tests", "cpp", "host_multi_file.cpp"),
                    "-L" + os.path.join(ROOT, "ngs_b200"), "-lngs_cuda", "-Wl,-rpath," + os.path.join(ROOT, "ngs_b200")], check=True)
    return out


DICT = [("chr1", 248956422), ("chr2", 242193529), ("chrM", 16569)]


def _dict(tmp_path, name, refs):
    p = tmp_path / name
    p.write_text("".join(f"{n} {l}\n" for n, l in refs))
    return str(p)


@pytest.mark.parametrize("case,other,index,there,here", [
    ("name", [("chr1", 248956422), ("chr3", 242193529), ("chrM", 16569)], 1, '"chr3" of length 242193529', '"chr2" of length 242193529'),
    ("length", [("chr1", 248956422), ("chr2", 242193528), ("chrM", 16569)], 1, '"chr2" of length 242193528', '"chr2" of length 242193529'),
    ("order", [("chr2", 242193529), ("chr1", 248956422), ("chrM", 16569)], 0, '"chr2" of length 242193529', '"chr1" of length 248956422'),
    ("fewer", DICT[:2], 2, "missing", '"chrM" of length 16569'),
    ("more", DICT + [("chrX", 156040895)], 3, '"chrX" of length 156040895', "missing"),
])
def test_a_different_dictionary_names_the_file_and_the_reference(exe, tmp_path, case, other, index, there, here):
    a, b = _dict(tmp_path, "first.txt", DICT), _dict(tmp_path, "second.txt", other)
    out = subprocess.run([exe, "dict", a, b], capture_output=True, text=True, check=True).stdout.strip()
    assert out == (f"error: the reference sequences of {b} differ from those of {a} ({len(other)} and {len(DICT)} references): "
                   f"reference {index} is {there} in {b} and {here} in {a}")
    assert subprocess.run([exe, "dict", a, _dict(tmp_path, "same.txt", DICT)], capture_output=True, text=True).stdout == "ok\n"


def _rows(out):
    return [[int(x) for x in ln.split()] for ln in out.splitlines()]


@pytest.mark.parametrize("n_dev,sizes,want", [
    (1, [5, 9, 1], [[1, 0, 2]]),
    (2, [5, 9, 1], [[1], [0, 2]]),
    (2, [4, 4, 4, 4], [[0, 2], [1, 3]]),                # ties: the lower index, the first of the least loaded
    (3, [10, 1, 1, 1, 1, 1, 1], [[0], [1, 3, 5], [2, 4, 6]]),
    (4, [7, 7, 7, 7], [[0], [1], [2], [3]]),
    (2, [1, 2, 3, 4, 5, 6], [[5, 2, 1], [4, 3, 0]]),
])
def test_whole_files_go_largest_first_to_the_least_loaded_device(exe, n_dev, sizes, want):
    out = subprocess.run([exe, "assign", str(n_dev)] + [str(s) for s in sizes], capture_output=True, text=True, check=True).stdout
    assert _rows(out) == want


@pytest.mark.parametrize("n_dev,sizes,want", [
    (4, [1, 1], [2, 2]),
    (4, [3, 1], [3, 1]),
    (8, [100, 1, 1], [6, 1, 1]),
    (5, [10, 10], [3, 2]),
    (8, [5, 3, 2, 1, 1, 1, 1], [2, 1, 1, 1, 1, 1, 1]),
    (3, [0, 0], [2, 1]),
])
def test_fewer_files_than_devices_share_them_by_size(exe, n_dev, sizes, want):
    out = subprocess.run([exe, "split", str(n_dev)] + [str(s) for s in sizes], capture_output=True, text=True, check=True).stdout
    got = _rows(out)[0]
    assert got == want and sum(got) == n_dev and min(got) >= 1


_S = {}


def _parts(kind, k):
    from ngs_b200 import ffi
    if "s" not in _S:
        _S["s"] = ffi.synth_bam(0, 20000, level=1)[0]
    return [bytes(f) for f in split_bam(_S["s"], k, kind, seed=3, block_payload=0x5300)]


@pytest.mark.parametrize("n_dev", [2, 4, 7])
@pytest.mark.parametrize("k", [1, 2, 3, 9])
@pytest.mark.parametrize("kind", SPLITS)
def test_the_plan_covers_every_record_once(exe, tmp_path, kind, k, n_dev):
    parts = _parts(kind, k)
    args, truths = [], []
    for i, raw in enumerate(parts):
        _, first, recs = walk(raw)
        p, t = tmp_path / f"f{i}.bam", tmp_path / f"t{i}.txt"
        p.write_bytes(raw)
        t.write_text("".join(f"{v} {r}\n" for v, r in recs))
        args += [str(p), str(first), str(t)]
        truths.append((first, recs))
    out = subprocess.run([exe, "plan", str(n_dev), "25"] + args, capture_output=True, text=True, check=True).stdout
    assert not out.startswith("error"), out
    lines = out.splitlines()
    queues = [[r[j:j + 4] for j in range(0, len(r), 4)] for r in _rows("\n".join(lines[:n_dev]))]
    cut, dropped = int(lines[n_dev].split()[1]), int(lines[n_dev + 1].split()[1])
    assert len(queues) == n_dev and all(queues)  # every device runs something
    assert cut == (k < n_dev)
    if not cut:
        assert dropped == 0
        assert sorted(p[0] for q in queues for p in q) == list(range(k))  # every file once, whole
        assert all(p[1:] == [truths[p[0]][0], 0, 0] for q in queues for p in q)
        return
    assert all(len(q) == 1 for q in queues)
    files = [q[0][0] for q in queues]
    assert files == sorted(files) and set(files) == set(range(k))  # every file at least one device, in file order
    assert sum(q[0][3] for q in queues) == dropped
    for f, (first, recs) in enumerate(truths):
        live = [q[0][1:3] for q in queues if q[0][0] == f and not q[0][3]]
        assert live[0][0] == first and live[-1][1] == 0
        assert all(a[1] == b[0] and a[0] < b[0] for a, b in zip(live, live[1:]))
        starts = {v for v, _ in recs}
        assert all(r[0] in starts for r in live[1:])  # every cut is a record start of that file
        bounds = [r[0] for r in live] + [1 << 64]
        assert [sum(1 for a, b in zip(bounds, bounds[1:]) if a <= v < b) for v, _ in recs] == [1] * len(recs)
