"""`qc` planned from a CSI (ngs_b200/host/bam.hpp: read_csi, parse_csi; the driver's app()): with only <BAM>.csi present the
results JSON is byte for byte the one planned from the file's .bai, a .bai wins over a .csi and a corrupt .csi alone fails
before any result is written; the plan cut inside contigs from a CSI, run shard by shard on one device, gives the oracle's
integers; and `qc --cuda-build-index --cuda-csi` writes the .csi `index --csi` and the oracle write, and nothing else."""
import gzip
import os
import subprocess

import numpy as np
import pytest

from baiutil import oracle_bai, unsorted_bams
from bamutil import EOF_BLOCK, bgzf_block
from csiutil import oracle_csi
from helpers import assert_same_ints, canonical_results, collect, merge_ints, oracle_ints
from test_host_csi_cpu import HTSLIB_SHAPES
from test_host_split_cpu import single_contig_bam

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "ngs_b200", "ngs-cuda-qc")
GRCH38 = "GRCh38_no_alt_AnalysisSet"
GC_SEED = 4


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count()
    except Exception:
        return 0


def _run(args):
    return subprocess.run([DRIVER] + args, capture_output=True, text=True)


def bgzf(payload):
    return b"".join(bgzf_block(payload[o:o + 0xFF00]) for o in range(0, len(payload), 0xFF00)) + EOF_BLOCK


_SYNTH = {}


def _synth(shape):
    from ngs_b200 import ffi
    if shape not in _SYNTH:
        bam, bai, info = ffi.synth_bam(shape, 3000 if shape == 2 else 40000, level=1)
        _SYNTH[shape] = (bam, bai, info)
    return _SYNTH[shape]


def _qc(path, outdir, prefix, *extra):
    r = _run(["qc", path, GRCH38, "-o", str(outdir), "-p", prefix, "--cuda-gc-seed", str(GC_SEED)] + list(extra))
    return r, os.path.join(str(outdir), prefix + ".results.json")


def _read(p):
    with open(p, "rb") as f:
        return f.read()


# ---------------------------------------------------------------- only a .csi
@pytest.mark.parametrize("shape", [0, 1, 2, 3])
def test_qc_from_a_csi_equals_qc_from_the_bai(shape, tmp_path):
    bam, bai, _ = _synth(shape)
    p = str(tmp_path / "x.bam")
    bam.tofile(p)
    with open(p + ".bai", "wb") as f:
        f.write(bytes(bai))
    r, want_json = _qc(p, tmp_path, "bai")
    assert r.returncode == 0, r.stderr
    want = _read(want_json)
    os.remove(p + ".bai")
    csis = {}
    for m in ("14", "16"):
        r = _run(["index", p, "--csi", "-m", m])
        assert r.returncode == 0, r.stderr
        csis["m" + m] = _read(p + ".csi")
        os.remove(p + ".csi")
    csis["htslib"] = bgzf(HTSLIB_SHAPES["all"](oracle_csi(bytes(bam), 14, 0)))
    for name, data in csis.items():
        with open(p + ".csi", "wb") as f:
            f.write(data)
        r, got = _qc(p, tmp_path, name)
        assert r.returncode == 0, (name, r.stderr)
        assert _read(got) == want, name
        assert not os.path.exists(p + ".bai")
        os.remove(p + ".csi")


def test_the_bai_wins_and_a_corrupt_csi_alone_fails(tmp_path):
    bam, bai, _ = _synth(3)
    p = str(tmp_path / "x.bam")
    bam.tofile(p)
    with open(p + ".bai", "wb") as f:
        f.write(bytes(bai))
    r, want_json = _qc(p, tmp_path, "bai")
    assert r.returncode == 0, r.stderr
    good = oracle_csi(bytes(bam), 14, 0)
    for name, data in (("magic", bgzf(b"CSJ\x01" + good[4:])), ("truncated", bgzf(good[:len(good) // 2])),
                       ("not_bgzf", gzip.compress(good)), ("empty", b"")):
        with open(p + ".csi", "wb") as f:
            f.write(data)
        r, got = _qc(p, tmp_path, "both_" + name)
        assert r.returncode == 0, (name, r.stderr)
        assert _read(got) == _read(want_json), name
        os.rename(p + ".bai", p + ".bai.aside")
        r, got = _qc(p, tmp_path, "csi_" + name)
        assert r.returncode != 0 and p + ".csi" in r.stderr, (name, r.stderr)
        assert not os.path.exists(got), name
        os.rename(p + ".bai.aside", p + ".bai")
    # neither index: the error of a missing .bai, as before
    os.remove(p + ".csi")
    os.remove(p + ".bai")
    r, got = _qc(p, tmp_path, "none")
    assert r.returncode != 0
    assert f"Could not find BAM index at {p}.bai. Please index the BAM first (`ngs index`)." in r.stderr
    assert not os.path.exists(got)


# ---------------------------------------------------------------- the split plan of a CSI, shard by shard on one device
@pytest.fixture(scope="module")
def host_csi(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("csi") / "host_csi")
    subprocess.run(["g++", "-O1", "-std=c++17", "-o", out, os.path.join(ROOT, "tests", "cpp", "host_csi.cpp"),
                    "-L" + os.path.join(ROOT, "ngs_b200"), "-lngs_cuda", "-Wl,-rpath," + os.path.join(ROOT, "ngs_b200")], check=True)
    return out


def csi_plan(exe, tmp_path, bam, payload, first, n_ref, k):
    """(shards as (first, end, empty, lo, hi, contigs), split) of the driver's plan_shards_split from the CSI payload"""
    b, c = tmp_path / "p.bam", tmp_path / "p.csi"
    b.write_bytes(bytes(bam))
    c.write_bytes(payload)
    out = subprocess.run([exe, str(b), str(c), "csi", str(first), str(n_ref), str(k)], capture_output=True, text=True,
                         check=True).stdout
    assert not out.startswith("error"), out
    shards, split = [], []
    for ln in out.splitlines():
        tag, *v = ln.split()
        if tag == "shard":
            v = [int(x) for x in v]
            shards.append((v[0], v[1], v[2], v[3], v[4], v[5:]))
        elif tag == "split":
            split = [int(x) for x in v]
    return shards, split


@pytest.mark.parametrize("k", [2, 3, 5, 8])
@pytest.mark.parametrize("shape", [0, 2, 3])
def test_csi_split_plan_on_one_device_equals_the_oracle(host_csi, tmp_path, shape, k):
    from ngs_b200 import ffi, formats
    from test_gpu_split import merge_split
    bam, bai, info = _synth(shape)
    want = oracle_ints(bam, bai, gc_seed=GC_SEED)
    b = np.ascontiguousarray(bam)
    plain = oracle_csi(bytes(bam), 14, 0)
    flags = ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_COVERAGE | ffi.NGSQ_F_VERIFY_CRC
    for name, payload in (("m14", plain), ("m16", oracle_csi(bytes(bam), 16, 0)), ("htslib", HTSLIB_SHAPES["all"](plain))):
        engines = [ffi.Engine(0, flags=flags, gc_seed=GC_SEED) for _ in range(k)]
        hdr = formats.read_header(engines[0], b)
        shards, split = csi_plan(host_csi, tmp_path, bam, payload, hdr.first_voffset, len(hdr.refs), k)
        assert len(shards) == k and sum(not s[2] for s in shards) > 1, name
        lens = [l for _, l in hdr.refs]
        enabled = [1 if formats.is_primary(n) else 0 for n, _ in hdr.refs]
        for e, (first, end, empty, lo, hi, _) in zip(engines, shards):
            e.set_references(lens, enabled)
            for c in split:
                e.split_reference(c)
            if empty:
                e.set_range(0, 0)
            else:
                e.set_range(first, end)
                e.submit(np.ascontiguousarray(b[lo:hi]), lo)
            e.finish()
        root = next((i for i, s in enumerate(shards) if any(c not in s[5] for c in split)), 0)
        merge_split(engines, split, root)
        got = merge_ints([collect(e, lens, enabled) for e in engines])
        assert sum(e.stats()["records"] for e in engines) == info["n_records"], name
        assert_same_ints(got, want)


# ---------------------------------------------------------------- --cuda-build-index --cuda-csi
def test_build_index_csi(tmp_path):
    bam, bai, _ = _synth(3)
    ref = str(tmp_path / "ref.bam")
    bam.tofile(ref)
    with open(ref + ".bai", "wb") as f:
        f.write(bytes(bai))
    r, plain_json = _qc(ref, tmp_path, "plain")
    assert r.returncode == 0, r.stderr
    for shift in (None, 16):
        tag = "default" if shift is None else f"m{shift}"
        p, q = str(tmp_path / f"{tag}.bam"), str(tmp_path / f"{tag}_index.bam")
        bam.tofile(p)
        bam.tofile(q)
        extra = ["--cuda-build-index", "--cuda-csi"] + ([] if shift is None else ["--cuda-min-shift", str(shift)])
        r, got = _qc(p, tmp_path, tag, *extra)
        assert r.returncode == 0, r.stderr
        assert not os.path.exists(p + ".bai")
        written = _read(p + ".csi")
        assert written.endswith(EOF_BLOCK)
        r = _run(["index", q, "--csi"] + ([] if shift is None else ["-m", str(shift)]))
        assert r.returncode == 0, r.stderr
        assert gzip.decompress(written) == gzip.decompress(_read(q + ".csi")) == oracle_csi(bytes(bam), shift or 14, 0)
        assert _read(got) == _read(plain_json)
        # the .csi is now the file's index: read and left as it is
        before = os.stat(p + ".csi").st_mtime_ns
        r, again = _qc(p, tmp_path, tag + "_again", *extra)
        assert r.returncode == 0, r.stderr
        assert os.stat(p + ".csi").st_mtime_ns == before and not os.path.exists(p + ".bai")
        assert _read(again) == _read(plain_json)
    # an existing .csi counts as the index for --cuda-build-index alone too
    r, again = _qc(str(tmp_path / "default.bam"), tmp_path, "bai_flag", "--cuda-build-index")
    assert r.returncode == 0, r.stderr
    assert not os.path.exists(str(tmp_path / "default.bam.bai"))


def test_build_index_csi_refusals(tmp_path):
    bam, _ = unsorted_bams()["position"]
    p = str(tmp_path / "u.bam")
    with open(p, "wb") as f:
        f.write(bytes(bam))
    r, got = _qc(p, tmp_path, "u", "--cuda-build-index", "--cuda-csi")
    assert r.returncode != 0 and "not coordinate-sorted" in r.stderr
    assert not os.path.exists(p + ".csi") and not os.path.exists(p + ".bai")
    for extra, match in ((["--cuda-csi"], "--cuda-build-index"), (["--cuda-build-index", "--cuda-min-shift", "16"], "--cuda-csi"),
                         (["--cuda-min-shift", "16"], "--cuda-csi"), (["--cuda-build-index", "--cuda-csi", "-n", "10"], "-n")):
        r, _ = _qc(p, tmp_path, "flags", *extra)
        assert r.returncode != 0 and match in r.stderr, (extra, r.stderr)
    assert not os.path.exists(p + ".csi") and not os.path.exists(p + ".bai")


# ---------------------------------------------------------------- several GPUs
@pytest.mark.parametrize("n", [2, 4])
def test_driver_on_distinct_devices(tmp_path, n):
    if _n_gpus() < n:
        pytest.skip(f"needs {n} GPUs")
    devs = ",".join(str(i) for i in range(n))
    bam, bai = single_contig_bam()  # one contig: every plan on several devices cuts inside it
    want_json = str(tmp_path / "o.json")
    oracle_ints(np.frombuffer(bam, dtype=np.uint8), np.frombuffer(bai, dtype=np.uint8), gc_seed=GC_SEED, json_path=want_json)
    p, q = str(tmp_path / "c.bam"), str(tmp_path / "b.bam")
    for path in (p, q):
        with open(path, "wb") as f:
            f.write(bam)
    with open(p + ".csi", "wb") as f:
        f.write(bgzf(oracle_csi(bam, 14, 0)))
    r, got = _qc(p, tmp_path, "multi", "--cuda-devices", devs)
    assert r.returncode == 0, r.stderr
    assert "Sharding inside contigs" in r.stderr
    assert canonical_results(got) == canonical_results(want_json)
    r, got = _qc(q, tmp_path, "built", "--cuda-devices", devs, "--cuda-build-index", "--cuda-csi")
    assert r.returncode == 0, r.stderr
    assert gzip.decompress(_read(q + ".csi")) == oracle_csi(bam, 14, 0) and not os.path.exists(q + ".bai")
    assert canonical_results(got) == canonical_results(want_json)
