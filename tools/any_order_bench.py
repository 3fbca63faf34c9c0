"""Measures `qc --cuda-any-order` (DESIGN.md section 5, "Records in any order") against `qc` on the same records sorted, on
bench.py's WGS shape (synthetic 2x150, the 25 GRCh38 primary contigs, zlib-1).  S is the sorted file with its .bai, U a copy
with the records in a seeded random order (tools/bamshuffle.cpp).  For each N of --gpus that the box has:

  * wall_ms_file_to_results: the driver's own figure (--cuda-perf: host clock from the first read to the results, the reduce
    included), median over --steps runs after --warmup, for S (its index's plan) and for U (--cuda-any-order), with the
    engine's per-stage times (CUDA events, the largest over ranks: `stages`) to show where a difference comes from;
  * ms_reduce: ngsq_reduce through the C ABI, one engine per GPU, max over ranks (CUDA events), for U cut at the driver's
    finder anchors with every reference split (every contig's int32 difference array and tile sums go through ncclReduce and
    the root resolves the whole genome), and for S cut contig-aligned (no split contig: one sum of the result buffers);
    reduce_bytes is what the split arrays put through ncclReduce per rank;
  * root_resolve_ms (on GPU 0 alone, so also on a one-GPU box): the root's share of that merge, K9 over every contig after
    the sum, timed on one engine that ran U whole with every reference split (ngsq_resolve_split; the kernels' cost does not
    depend on the values).

Two things here restate the driver and the engine rather than call them, and must be kept in step with them: anchor_cuts
is ngs_b200/host/bam.hpp's plan_shards_unindexed (the cuts the driver's any-order plan takes), and split_reduce_bytes is
bam.hpp's function of that name (the engine's int32 difference array and tile sums per contig).

U's results must equal S's apart from the GC window of reads longer than 101 bases (keyed by virtual offset, DESIGN.md
section 2).  The card's name and power limit are read in the same run.  Every file goes to a temporary directory, removed at
the end.  Prints one JSON line; --out writes it too.

  python tools/any_order_bench.py [--records N] [--steps K] [--warmup W] [--gpus 1,2,4,8] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
DRIVER = os.path.join(ROOT, "ngs_b200", "ngs-cuda-qc")
GRCH38 = "GRCh38_no_alt_AnalysisSet"
FIND_BLOCKS, FIND_BLOCKS_MAX = 4, 4096  # ngs_b200/host/bam.hpp: kFindBlocks, kFindBlocksMax
STAGES = ("ms_inflate", "ms_crc", "ms_scan", "ms_facets", "ms_coverage", "ms_tail", "ms_total")


def split_reduce_bytes(lens, enabled, split):
    """What the split arrays of `split` put through ncclReduce per rank (bam.hpp: split_reduce_bytes; Coverage's contigs)."""
    return int(sum((lens[c] + 2) * 4 + ((lens[c] + 4096) // 4096) * 4 + 8 for c in split if enabled[c]))


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "unknown"


def run_driver(path, outdir, tag, n, any_order):
    devs = ",".join(str(i) for i in range(n))
    args = [DRIVER, "qc", path, GRCH38, "-o", outdir, "-p", tag, "--cuda-perf", "--cuda-devices", devs] + (["--cuda-any-order"] if any_order else [])
    r = subprocess.run(args, capture_output=True, text=True)
    if r.returncode:
        raise SystemExit(f"driver failed: {' '.join(args)}\n{r.stderr}")
    perf = json.load(open(os.path.join(outdir, tag + ".perf.json")))
    plan = "any_order" if any_order else ("split" if "Sharding inside contigs" in r.stderr else "contig")
    return perf[0]["wall_ms_file_to_results"], {k: max(p[k] for p in perf) for k in STAGES}, plan


def anchor_cuts(finder, data, blocks, nb, first, n):
    """The driver's cuts (plan_shards_unindexed): targets snapped to the next block start, moved to the first record the
    finder sees from there; a cut that does not lie behind the previous one is left out."""
    base, size = first >> 16, data.size
    starts = [blocks[i].coffset for i in range(nb)]
    cuts = []
    for k in range(1, n):
        t = base + (size - base) * k // n
        j = next((i for i, c in enumerate(starts) if c >= t), nb)
        v, w = 0, FIND_BLOCKS
        while j < nb and w <= FIND_BLOCKS_MAX:
            last = min(j + w, nb) - 1
            hi = blocks[last].coffset + blocks[last].csize
            v, _ = finder.find_record(np.ascontiguousarray(data[starts[j]:hi]), starts[j])
            if v or last == nb - 1:
                break
            w *= 2
        if v and v > (cuts[-1] if cuts else first):
            cuts.append(v)
    return cuts


def run_reduce(engines, data, ranges, split, lens, enabled, blocks, nb, reduce=True):
    """One run of every engine over its range, then ngsq_reduce on all; returns (max ms_reduce, max ms_total)."""
    from ngs_b200 import formats
    errs = [None] * len(engines)

    def rank(i):
        try:
            e = engines[i]
            e.reset()
            e.set_references(lens, enabled)
            for c in split:
                e.split_reference(c)
            first, end = ranges[i] if i < len(ranges) else (0, 0)
            if first == 0:
                e.set_range(0, 0)
            else:
                lo, hi = formats.shard_byte_range(formats.Shard(first, end, []), blocks, nb, data.size)
                e.set_range(first, end)
                e.submit_ptr(data.ctypes.data + lo, hi - lo, lo)
            e.finish()
            if reduce:
                e.reduce(0)
        except Exception as ex:  # noqa: BLE001
            errs[i] = ex
    ts = [threading.Thread(target=rank, args=(i,)) for i in range(len(engines))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    for x in errs:
        if x:
            raise x
    st = [e.stats() for e in engines]
    return max(s["ms_reduce"] for s in st), max(s["ms_total"] for s in st)


def pinned_copy(lib, path):
    size = os.path.getsize(path)
    pin = lib.ngsq_host_alloc(size)
    data = np.ctypeslib.as_array(C.cast(pin, C.POINTER(C.c_uint8)), shape=(size,))
    data[:] = np.fromfile(path, dtype=np.uint8)
    return pin, data


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--records", type=int, default=20_000_000)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=1)
    p.add_argument("--gpus", default="1,2,4,8")
    p.add_argument("--out", default=None)
    args = p.parse_args()

    import torch
    from helpers import canonical_results
    from ngs_b200 import ffi, formats
    n_dev = torch.cuda.device_count()
    if n_dev < 1:
        raise SystemExit("any_order_bench needs a GPU")
    lib = ffi.load_library()
    tmp = tempfile.mkdtemp(prefix="any_order_bench_")
    try:
        s_path, u_path = os.path.join(tmp, "s.bam"), os.path.join(tmp, "u.bam")
        bam, bai, info = ffi.synth_bam(1, args.records, level=1)
        bam.tofile(s_path)
        bai.tofile(s_path + ".bai")
        del bam
        exe = os.path.join(tmp, "bamshuffle")
        subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tools", "bamshuffle.cpp"), "-lz", "-lpthread"], check=True)
        subprocess.run([exe, s_path, u_path, "7", "1"], check=True, capture_output=True)
        out = {"metric": "qc of a file in any order (--cuda-any-order) against the same records sorted", "card": card(),
               "gpus_present": n_dev, "records": info["n_records"], "compressed_bytes_sorted": os.path.getsize(s_path),
               "compressed_bytes_any_order": os.path.getsize(u_path), "steps": args.steps, "warmup": args.warmup, "runs": [],
               "unmeasured": []}
        ns = [int(x) for x in args.gpus.split(",")]
        for n in ns:
            if n > n_dev:
                out["unmeasured"].append(n)
                continue
            row = {"n": n}
            for name, path, any_order in (("sorted", s_path, False), ("any_order", u_path, True)):
                walls, stages = [], []
                for it in range(args.warmup + args.steps):
                    wall, st, plan = run_driver(path, tmp, f"{name}{n}", n, any_order)
                    if it >= args.warmup:
                        walls.append(wall)
                        stages.append(st)
                row[name] = {"plan": plan, "wall_ms_file_to_results": float(np.median(walls)),
                             "stages": {k: float(np.median([st[k] for st in stages])) for k in STAGES}}
            got, want = canonical_results(os.path.join(tmp, f"any_order{n}.results.json")), canonical_results(os.path.join(tmp, f"sorted{n}.results.json"))
            g, w = got.pop("gc_content"), want.pop("gc_content")
            row["results_equal_except_gc_window"] = got == want and g["records"] == w["records"]
            out["runs"].append(row)
            print(json.dumps(row), file=sys.stderr)
        # ngsq_reduce through the C ABI
        flags = ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_COVERAGE | ffi.NGSQ_F_VERIFY_CRC
        finder = ffi.Engine(0, flags=flags)
        for name, path in (("sorted", s_path), ("any_order", u_path)):
            pin, data = pinned_copy(lib, path)
            blocks, nb, _ = ffi.bgzf_walk(data)
            hdr = formats.read_header(finder, data)
            lens = [l for _, l in hdr.refs]
            enabled = [1 if formats.is_primary(x) else 0 for x, _ in hdr.refs]
            if name == "any_order":
                times = []
                for it in range(args.warmup + args.steps):
                    run_reduce([finder], data, [(hdr.first_voffset, 0)], list(range(len(lens))), lens, enabled, blocks, nb, reduce=False)
                    t0 = time.perf_counter()
                    finder.resolve_split(True)  # ends in a device synchronise
                    if it >= args.warmup:
                        times.append((time.perf_counter() - t0) * 1e3)
                out["root_resolve_ms"] = float(np.median(times))
                out["reduce_bytes_per_rank_any_order"] = split_reduce_bytes(lens, enabled, range(len(lens)))
            for row in out["runs"]:
                n = row["n"]
                if n < 2:
                    continue
                if name == "sorted":
                    shards = formats.plan_shards(hdr, formats.parse_bai(open(s_path + ".bai", "rb").read()), n, data.size)
                    ranges = [(0, 0) if s.first_voffset == 0 and not s.contigs else (s.first_voffset, s.end_voffset) for s in shards]
                    split = []
                else:
                    finder.reset()
                    finder.set_references(lens, [0] * len(lens))
                    cuts = anchor_cuts(finder, data, blocks, nb, hdr.first_voffset, n)
                    bounds = [hdr.first_voffset] + cuts
                    ranges = [(b, bounds[i + 1] if i + 1 < len(bounds) else 0) for i, b in enumerate(bounds)]
                    split = list(range(len(lens)))
                engines = [ffi.Engine(d, flags=flags) for d in range(n)]
                uid = ffi.nccl_unique_id()
                ts = [threading.Thread(target=engines[i].comm_init, args=(n, i, uid)) for i in range(n)]
                for t in ts:
                    t.start()
                for t in ts:
                    t.join()
                rs = [run_reduce(engines, data, ranges, split, lens, enabled, blocks, nb) for _ in range(args.warmup + args.steps)][args.warmup:]
                row[name]["ms_reduce"] = float(np.median([r[0] for r in rs]))
                row[name]["reduce_bytes"] = split_reduce_bytes(lens, enabled, split)
                for e in engines:
                    e.close()
            lib.ngsq_host_free(pin)
        finder.close()
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
