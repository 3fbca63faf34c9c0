"""Measures multi-GPU `qc` with contig-aligned shards against shards cut inside contigs (DESIGN.md section 5) on four synthetic
files: shape 0 (chr1, chr2, chrM), shape 1 (the 25-contig WGS shape), shape 2 (long reads, chr1-chr5) and shape 0 reduced to
chr1 (a single-contig file).  For N = 2, 4, 8 shards and each plan (formats.plan_shards / plan_shards_split), as the median over
--steps runs after --warmup:

  * shard_ms / device_ms: every shard run alone on GPU 0, one after the other (the engine's ms_total, CUDA events); device_ms
    is the slowest shard plus, for the split plan, root_resolve_ms.  This is what N GPUs would spend before the merge,
    measured on one;
  * root_resolve_ms: the root's resolve of the split contigs after the merge (K9 over every split contig, touched), timed on an
    engine that ran the whole file with the split set declared (the kernels' cost does not depend on the values);
  * reduce_bytes: what the split-array ncclReduce moves per rank (int32 difference arrays and tile sums, touched words);
  * with N GPUs present, also the real run: one engine per GPU and ngsq_reduce, nccl_wall_ms (host clock from the first
    submit to the end of the last rank's ngsq_reduce; setup is outside it), nccl_device_ms (max over ranks of ms_total +
    ms_reduce) and nccl_reduce_ms (max over ranks of ms_reduce, which includes the split-array reduce and the root's
    resolve).

The root's integers of the two plans must be equal.  The card's name and power limit are read in the same run.  Prints one
JSON line; --out writes it too.

  python tools/split_bench.py [--records N] [--records-long N] [--steps K] [--warmup W] [--gpus 2,4,8] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_name_and_power():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "unknown"


def setup(engines, shards, split, lens, enabled):
    for e in engines:
        e.reset()
        e.set_references(lens, enabled)
        for c in split:
            e.split_reference(c)


def submit_shard(e, s, data, blocks, nb):
    from ngs_b200 import formats
    if s.first_voffset == 0 and not s.contigs:
        e.set_range(0, 0)
    else:
        lo, hi = formats.shard_byte_range(s, blocks, nb, data.size)
        e.set_range(s.first_voffset, s.end_voffset)
        e.submit_ptr(data.ctypes.data + lo, hi - lo, lo)
    e.finish()


def run_nccl(engines, data, shards, split, lens, enabled, blocks, nb):
    setup(engines, shards, split, lens, enabled)
    errs = [None] * len(engines)

    def rank(i):
        try:
            submit_shard(engines[i], shards[i], data, blocks, nb)
            engines[i].reduce(0)
        except Exception as ex:  # noqa: BLE001
            errs[i] = ex
    t0 = time.perf_counter()
    ts = [threading.Thread(target=rank, args=(i,)) for i in range(len(engines))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    wall = (time.perf_counter() - t0) * 1e3
    for x in errs:
        if x:
            raise x
    st = [e.stats() for e in engines]
    return wall, max(s["ms_total"] + s["ms_reduce"] for s in st), max(s["ms_reduce"] for s in st)


def run_shards_on_one(e, data, shards, split, lens, enabled, blocks, nb):
    """Every shard alone on e's GPU, one after the other: the ms_total of each."""
    out = []
    for s in shards:
        setup([e], shards, split, lens, enabled)
        submit_shard(e, s, data, blocks, nb)
        out.append(e.stats()["ms_total"])
    return out


def root_resolve_ms(e, data, hdr, split, lens, enabled, blocks, nb):
    from ngs_b200 import formats
    whole = formats.Shard(hdr.first_voffset, 0, list(range(len(lens))))
    setup([e], [whole], split, lens, enabled)
    submit_shard(e, whole, data, blocks, nb)
    t0 = time.perf_counter()
    e.resolve_split(True)  # ends in a device synchronise
    return (time.perf_counter() - t0) * 1e3


def reduce_bytes(split, lens, enabled):
    return int(sum((lens[c] + 2) * 4 + ((lens[c] + 4096) // 4096) * 4 + 8 for c in split if enabled[c]))


def root_ints(e, lens, enabled):
    from helpers import collect
    out = collect(e, lens, enabled)
    out.pop("stats")
    return out


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--records", type=int, default=20_000_000, help="records of the short-read files")
    p.add_argument("--records-long", type=int, default=400_000, help="records of the long-read file")
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=1)
    p.add_argument("--gpus", default="2,4,8")
    p.add_argument("--out", default=None)
    args = p.parse_args()

    import torch
    from helpers import assert_same_ints
    from ngs_b200 import ffi, formats
    n_dev = torch.cuda.device_count()
    if n_dev < 1:
        raise SystemExit("split_bench needs a GPU")
    lib = ffi.load_library()
    files = [("shape0", 0, args.records, None), ("wgs_shape1", 1, args.records, None), ("shape2", 2, args.records_long, None),
             ("single_contig", 0, args.records, 1)]
    out = {"card": gpu_name_and_power(), "gpus_present": n_dev, "steps": args.steps, "warmup": args.warmup, "runs": []}
    flags = ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_COVERAGE | ffi.NGSQ_F_VERIFY_CRC
    one = ffi.Engine(0, flags=flags)
    for name, shape, n_rec, mask in files:
        bam, bai, info = ffi.synth_bam(shape, n_rec, level=1, **({"contig_mask": mask} if mask else {}))
        size = int(bam.size)
        pin = lib.ngsq_host_alloc(size)
        data = np.ctypeslib.as_array(C.cast(pin, C.POINTER(C.c_uint8)), shape=(size,))
        data[:] = bam
        del bam
        blocks, nb, _ = ffi.bgzf_walk(data)
        bai_p = formats.parse_bai(bai.tobytes())
        hdr = formats.read_header(one, data)
        lens = [l for _, l in hdr.refs]
        enabled = [1 if formats.is_primary(x) else 0 for x, _ in hdr.refs]
        for n in [int(x) for x in args.gpus.split(",")]:
            engines = None
            if n <= n_dev:
                engines = [ffi.Engine(d, flags=flags) for d in range(n)]
                uid = ffi.nccl_unique_id()
                ts = [threading.Thread(target=engines[i].comm_init, args=(n, i, uid)) for i in range(n)]
                for t in ts:
                    t.start()
                for t in ts:
                    t.join()
            results = {}
            for plan in ("contig", "split"):
                if plan == "contig":
                    shards, split = formats.plan_shards(hdr, bai_p, n, size), []
                else:
                    shards, split = formats.plan_shards_split(hdr, bai_p, n, size)
                per = []
                for s in shards:
                    if s.first_voffset == 0 and not s.contigs:
                        per.append(0)
                    else:
                        lo, hi = formats.shard_byte_range(s, blocks, nb, size)
                        per.append(hi - lo)
                rows = []
                for it in range(args.warmup + args.steps):
                    r = run_shards_on_one(one, data, shards, split, lens, enabled, blocks, nb)
                    if it >= args.warmup:
                        rows.append(r)
                shard_ms = [float(np.median([r[i] for r in rows])) for i in range(len(shards))]
                resolve = float(np.median([root_resolve_ms(one, data, hdr, split, lens, enabled, blocks, nb)
                                           for _ in range(args.steps)])) if split else 0.0
                run = {"file": name, "records": info["n_records"], "n": n, "plan": plan, "split": split, "shard_bytes": per,
                       "shard_ms": shard_ms, "root_resolve_ms": resolve, "device_ms": max(shard_ms) + resolve,
                       "reduce_bytes": reduce_bytes(split, lens, enabled)}
                if engines:
                    nr = [run_nccl(engines, data, shards, split, lens, enabled, blocks, nb) for _ in range(args.warmup + args.steps)]
                    nr = nr[args.warmup:]
                    run.update(nccl_wall_ms=float(np.median([r[0] for r in nr])), nccl_device_ms=float(np.median([r[1] for r in nr])),
                               nccl_reduce_ms=float(np.median([r[2] for r in nr])))
                    results[plan] = root_ints(engines[0], lens, enabled)
                out["runs"].append(run)
                print(json.dumps(run), file=sys.stderr)
            if engines:
                assert_same_ints(results["split"], results["contig"])
                for e in engines:
                    e.close()
        lib.ngsq_host_free(pin)
    one.close()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
