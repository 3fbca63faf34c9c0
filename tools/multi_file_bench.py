"""Measures `qc --cuda-also` (DESIGN.md section 5, "Several files") on bench.py's WGS shape (synthetic 2x150, the 25 GRCh38
primary contigs, zlib-1).  S is the sorted file with its .bai; for each K of --parts, S's records are written again as K files of
consecutive records, each with S's header, the way a basecaller writes one sample as chunk files (tools/bamshuffle.cpp, seed 0).
On GPU 0, for each K:

  * also: one driver invocation over the K files (`--cuda-also`; for K = 1 the one file with `--cuda-any-order`, the same
    rules), median over --steps runs after --warmup: the process's wall clock (host clock around the subprocess: start, CUDA
    context, engine allocations, the headers, the pass, the JSON) and the driver's wall_ms_file_to_results (--cuda-perf: first
    read to results), with the engine's per-stage times (CUDA events);
  * loop: a separate invocation per file (`--cuda-any-order`), one after the other, as a user without the flag runs them: the
    wall clock of the loop over the first min(K, --loop-max) files, and per invocation.  Its per-file JSONs cannot be merged
    into the sample's results (the depth histogram and its derived values are no sums); only the time is of interest.

S itself goes through the driver once per step as the reference point (`sorted`).  The results of every `--cuda-also` run must
equal S's, apart from the GC window of reads longer than 101 bases, which is keyed by virtual offset in each file.  The card's
name and power limit are read in the same run.  Every file goes to a temporary directory, removed at the end.  Prints one JSON
line; --out writes it too.

  python tools/multi_file_bench.py [--records N] [--parts 1,8,64,512] [--steps K] [--warmup W] [--loop-max M] [--out FILE]
"""
import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

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


def run_driver(paths, outdir, tag, extra):
    also = [a for p in paths[1:] for a in ("--cuda-also", p)]
    args = [DRIVER, "qc", paths[0], GRCH38, "-o", outdir, "-p", tag, "--cuda-perf"] + also + extra
    t0 = time.perf_counter()
    r = subprocess.run(args, capture_output=True, text=True)
    wall = (time.perf_counter() - t0) * 1e3
    if r.returncode:
        raise SystemExit(f"driver failed: {' '.join(args[:8])} ..\n{r.stderr}")
    perf = json.load(open(os.path.join(outdir, tag + ".perf.json")))[0]
    return wall, perf


def timed(paths, outdir, tag, extra, steps, warmup):
    walls, perfs = [], []
    for it in range(warmup + steps):
        wall, perf = run_driver(paths, outdir, tag, extra)
        if it >= warmup:
            walls.append(wall)
            perfs.append(perf)
    return {"process_wall_ms": float(np.median(walls)), "process_wall_ms_runs": walls,
            "wall_ms_file_to_results": float(np.median([p["wall_ms_file_to_results"] for p in perfs])),
            "stages": {k: float(np.median([p[k] for p in perfs])) for k in STAGES},
            "files_on_device": perfs[0].get("files", 1)}


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--records", type=int, default=20_000_000)
    p.add_argument("--parts", default="1,8,64,512")
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=1)
    p.add_argument("--loop-max", type=int, default=64)
    p.add_argument("--out", default=None)
    args = p.parse_args()

    import torch
    from helpers import canonical_results
    from ngs_b200 import ffi
    if torch.cuda.device_count() < 1:
        raise SystemExit("multi_file_bench needs a GPU")
    tmp = tempfile.mkdtemp(prefix="multi_file_bench_")
    try:
        s_path = os.path.join(tmp, "s.bam")
        bam, bai, info = ffi.synth_bam(1, args.records, level=1)
        bam.tofile(s_path)
        bai.tofile(s_path + ".bai")
        del bam
        exe = os.path.join(tmp, "bamshuffle")
        subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tools", "bamshuffle.cpp"), "-lz", "-lpthread"], check=True)
        out = {"metric": "qc of one sample in K files: one --cuda-also invocation, the driver on the one sorted file, and one invocation per file",
               "card": card(), "records": info["n_records"], "compressed_bytes_sorted": os.path.getsize(s_path), "steps": args.steps,
               "warmup": args.warmup, "sorted": timed([s_path], tmp, "sorted", [], args.steps, args.warmup), "runs": []}
        print(json.dumps({"sorted": out["sorted"]}), file=sys.stderr)
        want = canonical_results(os.path.join(tmp, "sorted.results.json"))
        want.pop("gc_content")
        for k in [int(x) for x in args.parts.split(",")]:
            d = os.path.join(tmp, f"k{k}")
            os.makedirs(d)
            subprocess.run([exe, s_path, os.path.join(d, "one.bam" if k == 1 else "part"), "0", "1", str(os.cpu_count() or 1), str(k)],
                           check=True, capture_output=True)
            paths = [os.path.join(d, "one.bam")] if k == 1 else [os.path.join(d, f"part.{i}.bam") for i in range(k)]
            row = {"parts": k, "compressed_bytes": sum(os.path.getsize(x) for x in paths),
                   "also": timed(paths, d, "also", ["--cuda-any-order"] if k == 1 else [], args.steps, args.warmup)}
            got = canonical_results(os.path.join(d, "also.results.json"))
            got.pop("gc_content")
            row["results_equal_except_gc_window"] = got == want
            n_loop = min(k, args.loop_max)
            t0 = time.perf_counter()
            for i in range(n_loop):
                run_driver([paths[i]], d, f"one{i}", ["--cuda-any-order"])
            loop = (time.perf_counter() - t0) * 1e3
            row["loop"] = {"files_timed": n_loop, "wall_ms": loop, "wall_ms_per_invocation": loop / n_loop}
            out["runs"].append(row)
            print(json.dumps(row), file=sys.stderr)
            shutil.rmtree(d, ignore_errors=True)
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
