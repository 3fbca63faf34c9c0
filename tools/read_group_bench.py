"""Measures `qc --cuda-by-read-group` (DESIGN.md section 5, "Read groups") on bench.py's WGS shape (synthetic 2x150, the 25
GRCh38 primary contigs, zlib-1) and on the long-read shape (c4).  For each K, the driver runs with the flag and without it on
the same file, median over --steps runs after --warmup: the process's wall clock (host clock around the subprocess) and the
driver's wall_ms_file_to_results (--cuda-perf), with the engine's per-stage times (CUDA events; the read-group kernels run
inside ms_facets).

The generator writes up to 10 read groups (rg0..rg9, from bits of each record's random draw).  For K <= 10 the file is the
generator's, sorted, with its .bai.  For K > 10 its header is written again with K @RG lines (the records still carry rg0..rg9,
so K - 10 groups stay empty but hold their tables) and both runs take `--cuda-any-order`, since the .bai no longer matches the
file's offsets.  The card's name and power limit are read in the same run.  Every file goes to a temporary directory, removed at
the end.  Prints one JSON line; --out writes it too.

  python tools/read_group_bench.py [--records N] [--groups 1,8,64,512] [--long-records N] [--steps K] [--warmup W] [--out FILE]
"""
import argparse
import json
import os
import shutil
import struct
import subprocess
import sys
import tempfile
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
DRIVER = os.path.join(ROOT, "ngs_b200", "ngs-cuda-qc")
GRCH38 = "GRCh38_no_alt_AnalysisSet"
STAGES = ("ms_inflate", "ms_crc", "ms_scan", "ms_facets", "ms_coverage", "ms_tail", "ms_total", "waves")


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "unknown"


def run_driver(path, outdir, tag, extra):
    args = [DRIVER, "qc", path, GRCH38, "-o", outdir, "-p", tag, "--cuda-perf"] + extra
    t0 = time.perf_counter()
    r = subprocess.run(args, capture_output=True, text=True)
    wall = (time.perf_counter() - t0) * 1e3
    if r.returncode:
        raise SystemExit(f"driver failed: {' '.join(args)}\n{r.stderr}")
    return wall, json.load(open(os.path.join(outdir, tag + ".perf.json")))[0]


def timed(path, outdir, tag, extra, steps, warmup):
    walls, perfs = [], []
    for it in range(warmup + steps):
        wall, perf = run_driver(path, outdir, tag, extra)
        if it >= warmup:
            walls.append(wall)
            perfs.append(perf)
    return {"process_wall_ms": float(np.median(walls)), "process_wall_ms_runs": walls,
            "wall_ms_file_to_results": float(np.median([p["wall_ms_file_to_results"] for p in perfs])),
            "stages": {k: float(np.median([p[k] for p in perfs])) for k in STAGES}}


def with_groups(bam: bytes, k: int) -> bytes:
    """The file with its header written again with @RG lines rg0..rg{k-1} (the generator keeps the header in blocks of its own)."""
    from bamutil import bgzf_block
    off, hdr = 0, b""
    while True:
        bsize = int.from_bytes(bam[off + 16:off + 18], "little") + 1
        hdr += zlib.decompress(bam[off + 18:off + bsize - 8], -15)
        off += bsize
        l_text = int.from_bytes(hdr[4:8], "little")
        if len(hdr) >= 12 + l_text:
            p, n_ref = 12 + l_text, int.from_bytes(hdr[8 + l_text:12 + l_text], "little")
            for _ in range(n_ref):
                if p + 4 > len(hdr):
                    break
                p += 8 + int.from_bytes(hdr[p:p + 4], "little")
            else:
                if p == len(hdr):
                    break
    l_text = int.from_bytes(hdr[4:8], "little")
    text = hdr[8:8 + l_text].decode()
    lines = [ln for ln in text.split("\n") if ln and not ln.startswith("@RG")]
    text = "\n".join(lines[:-1] + [f"@RG\tID:rg{i}\tSM:synthetic" for i in range(k)] + lines[-1:]) + "\n"
    new = b"BAM\x01" + struct.pack("<i", len(text)) + text.encode() + hdr[8 + l_text:]
    out = b"".join(bgzf_block(new[o:o + 0xFF00], 1) for o in range(0, len(new), 0xFF00))
    return out + bam[off:]


def measure(path, d, groups, extra, steps, warmup):
    row = {"groups_declared": groups, "without": timed(path, d, "plain", extra, steps, warmup),
           "with": timed(path, d, "rg", extra + ["--cuda-by-read-group"], steps, warmup)}
    row["extra_ms_facets"] = row["with"]["stages"]["ms_facets"] - row["without"]["stages"]["ms_facets"]
    row["extra_wall_ms_file_to_results"] = row["with"]["wall_ms_file_to_results"] - row["without"]["wall_ms_file_to_results"]
    row["extra_process_wall_ms"] = row["with"]["process_wall_ms"] - row["without"]["process_wall_ms"]
    row["sample_json_identical"] = open(os.path.join(d, "plain.results.json"), "rb").read() == open(os.path.join(d, "rg.results.json"), "rb").read()
    return row


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--records", type=int, default=20_000_000)
    p.add_argument("--groups", default="1,8,64,512")
    p.add_argument("--long-records", type=int, default=200_000)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=1)
    p.add_argument("--out", default=None)
    args = p.parse_args()

    import torch
    from ngs_b200 import ffi
    if torch.cuda.device_count() < 1:
        raise SystemExit("read_group_bench needs a GPU")
    tmp = tempfile.mkdtemp(prefix="read_group_bench_")
    try:
        out = {"metric": "qc --cuda-by-read-group against the same run without the flag (medians)", "card": card(),
               "records": args.records, "steps": args.steps, "warmup": args.warmup, "wgs": [], "long_read": None}
        for k in [int(x) for x in args.groups.split(",")]:
            d = os.path.join(tmp, f"k{k}")
            os.makedirs(d)
            bam, bai, info = ffi.synth_bam(1, args.records, level=1, read_groups=min(k, 10))
            path = os.path.join(d, "s.bam")
            if k <= 10:
                bam.tofile(path)
                bai.tofile(path + ".bai")
                extra = []
            else:
                with open(path, "wb") as f:
                    f.write(with_groups(bam.tobytes(), k))
                extra = ["--cuda-any-order"]
            del bam
            row = measure(path, d, k, extra, args.steps, args.warmup)
            row.update(records_in_groups=min(k, 10), any_order=bool(extra), compressed_bytes=os.path.getsize(path))
            out["wgs"].append(row)
            print(json.dumps(row), file=sys.stderr)
            shutil.rmtree(d, ignore_errors=True)
        d = os.path.join(tmp, "c4")
        os.makedirs(d)
        bam, bai, info = ffi.synth_bam(2, args.long_records, level=1, read_groups=8)
        path = os.path.join(d, "s.bam")
        bam.tofile(path)
        bai.tofile(path + ".bai")
        del bam
        out["long_read"] = measure(path, d, 8, [], args.steps, args.warmup)
        out["long_read"]["records"] = info["n_records"]
        print(json.dumps(out["long_read"]), file=sys.stderr)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
