"""Measures the GPU BAI build (NGSQ_F_INDEX) on bench.py's default workload: the same 2x150bp WGS-shaped synthetic BAM (bench
seed, shape and zlib level; 100 M records unless --records), indexed

  * resident: the compressed file in HBM, ngsq_submit_device + ngsq_finish + ngsq_get_bai, index only;
  * end to end: ngsq_submit from pinned host memory in --chunk-mb chunks, index only;
  * beside qc: bench.py's resident qc step (record facets + coverage + CRC) with and without NGSQ_F_INDEX, alternated.

Device times are the engine's CUDA-event totals (ms_total); wall times are host clocks around calls that end in a device
synchronise and include the host's assembly of the .bai.  The result is compared with the oracle's single-thread index of
the same file (tests/cpp/bai_oracle.c, a restatement of the reference's `ngs index` loop over zlib; its time is the CPU
baseline) and with bamgen's (equal up to bamgen's clamped linear index).  Prints one JSON line; --out writes it too.

--gpus N measures the index of a file without an index cut between N devices instead (NGSQ_F_INDEX_PART): cuts by the
driver's rule (targets snapped to the next block start, anchors from ngsq_find_record), one engine and one host thread per
device, each part's compressed bytes resident on its device (resident) or streamed from pinned host memory (end to end); the
step is the slowest thread, and the host's ngsq_join_bai is timed on its own.  The joined .bai must equal one NGSQ_F_INDEX
engine's and the oracle's byte for byte.

--driver compares the host driver on a file: `qc --cuda-build-index` (one read) against `index` then `qc` (two reads), wall
time per command sequence, alternated.  The driver reads with O_DIRECT, so the page cache does not serve the file.

--csi compares the CSI build (NGSQ_F_INDEX_CSI, min_shift 14, depth 5 on this workload) with the BAI build on the same
file: index-only device time resident and end to end, the two engines alternated; the host assembly of each format, timed
as the join of one part (ngsq_join_bai / ngsq_join_csi over a single NGSQ_F_INDEX_PART engine: the run sort, the chunks,
the windows and the serialiser); then the CSI of bamgen shape 4 (references of 1.9 and 0.8 Gbp) at --shape4-records.  Both
payloads must equal the oracle's (unless --no-oracle).

  python tools/index_bench.py [--records N] [--steps K] [--warmup W] [--chunk-mb M] [--no-oracle] [--gpus N | --driver | --csi]
                              [--shape4-records N] [--out FILE]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_name_and_power():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return r.stdout.strip() if r.returncode == 0 else "unknown"


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--records", type=int, default=0, help="records (default: bench.py's wgs size, 100 M)")
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=2)
    p.add_argument("--chunk-mb", type=int, default=256)
    p.add_argument("--no-oracle", action="store_true", help="skip the single-thread oracle index (minutes on 100 M records)")
    p.add_argument("--gpus", type=int, default=0, help="index parts on N devices (0: the one-engine measurements)")
    p.add_argument("--driver", action="store_true", help="qc --cuda-build-index against index + qc, from a file")
    p.add_argument("--csi", action="store_true", help="CSI against BAI on the workload, then CSI on bamgen shape 4")
    p.add_argument("--shape4-records", type=int, default=20_000_000)
    p.add_argument("--out", default=None)
    args = p.parse_args()

    import torch
    import bench
    from ngs_b200 import ffi, formats
    from baiutil import oracle_bai

    wl = bench.workload("wgs", 1, args.records, -1)
    mask, with_tail = bench.workload_shard(wl, 0)
    t0 = time.perf_counter()
    bam, bai_writer, info = ffi.synth_bam(wl["shape"], wl["total_records"], level=wl["level"], contig_mask=mask, with_tail=with_tail)
    gen_s = time.perf_counter() - t0
    n_rec, C_bytes, D_bytes = info["n_records"], int(bam.size), int(info["inflated_bytes"])
    print(f"generated {n_rec} records, {C_bytes} bytes in {gen_s:.1f} s", file=sys.stderr)

    if args.driver:
        return driver_bench(args, bam, bai_writer, n_rec)
    lib = ffi.load_library()
    pin = lib.ngsq_host_alloc(C_bytes)
    pinned = np.ctypeslib.as_array(C.cast(pin, C.POINTER(C.c_uint8)), shape=(C_bytes,))
    pinned[:] = bam
    del bam
    blocks, n_blocks, used = ffi.bgzf_walk(pinned)
    assert used == C_bytes
    d_comp = torch.empty(C_bytes + 512, dtype=torch.uint8, device="cuda")
    d_comp[:C_bytes].copy_(torch.from_numpy(pinned))
    torch.cuda.synchronize()
    cuts = [0]
    acc = 0
    for i in range(n_blocks):
        acc += blocks[i].csize
        if acc - cuts[-1] >= args.chunk_mb << 20:
            cuts.append(acc)
    if cuts[-1] != C_bytes:
        cuts.append(C_bytes)

    if args.gpus:
        return parts_bench(args, pinned, pin, blocks, n_blocks, n_rec, C_bytes, D_bytes, d_comp, lib)
    if args.csi:
        return csi_bench(args, pinned, pin, blocks, n_blocks, n_rec, C_bytes, D_bytes, d_comp, cuts, wl, lib)

    def engine(flags):
        e = ffi.Engine(flags=flags, gc_seed=bench.GC_SEED, reserve_compressed=C_bytes, reserve_inflated=D_bytes + 65536, reserve_blocks=n_blocks + 16)
        hdr = formats.read_header(e, pinned)
        e.set_references([l for _, l in hdr.refs], [1 if formats.is_primary(nm) else 0 for nm, _ in hdr.refs])
        e.set_range(hdr.first_voffset, 0)
        return e

    def resident(e, bai=False):
        t = time.perf_counter()
        e.reset()
        e.submit_device(d_comp.data_ptr(), C_bytes, blocks, n_blocks)
        e.finish()
        out = e.bai() if bai else None
        return (time.perf_counter() - t) * 1e3, e.stats()["ms_total"], out

    def e2e(e):
        t = time.perf_counter()
        e.reset()
        for a, b in zip(cuts[:-1], cuts[1:]):
            if b == C_bytes:
                e.flush()
            e.submit_ptr(pin + a, b - a, a)
        e.finish()
        out = e.bai()
        return (time.perf_counter() - t) * 1e3, e.stats()["ms_total"], out

    crc = ffi.NGSQ_F_VERIFY_CRC
    ix = engine(ffi.NGSQ_F_INDEX | crc)
    for _ in range(args.warmup):
        resident(ix, True)
    res = [resident(ix, True) for _ in range(args.steps)]
    gpu_bai = res[-1][2]
    assert all(r[2] == gpu_bai for r in res)
    ix_stats = ix.stats()
    for _ in range(max(1, args.warmup // 2)):
        e2e(ix)
    ee = [e2e(ix) for _ in range(args.steps)]
    assert all(r[2] == gpu_bai for r in ee)
    ix.close()

    qc_flags = ffi.NGSQ_F_RECORD_FACETS | ffi.NGSQ_F_COVERAGE | crc
    qc, qcx = engine(qc_flags), engine(qc_flags | ffi.NGSQ_F_INDEX)
    for _ in range(args.warmup):
        resident(qc)
        resident(qcx, True)
    plain, with_ix = [], []
    for _ in range(args.steps):  # alternated: other tenants of the host shift both sides alike
        plain.append(resident(qc))
        with_ix.append(resident(qcx, True))
    assert with_ix[-1][2] == gpu_bai
    qc.close()
    qcx.close()
    del d_comp
    torch.cuda.synchronize()

    med = lambda xs: float(np.median(xs))  # noqa: E731
    parsed = formats.parse_bai(gpu_bai)
    chunks = sum(len(c) for r in parsed.refs for c in r.bins.values())
    # bamgen's index: equal but for its linear index clamped to L >> 14
    want = formats.parse_bai(bai_writer.tobytes())
    same_as_bamgen = parsed.n_no_coor == want.n_no_coor and all(
        list(g.bins.items()) == list(w.bins.items()) and (g.ref_beg, g.ref_end, g.n_mapped, g.n_unmapped) == (w.ref_beg, w.ref_end, w.n_mapped, w.n_unmapped)
        and g.linear[: len(w.linear)] == w.linear for g, w in zip(parsed.refs, want.refs))
    out = {
        "metric": "BAI build records/sec (resident, index only, device)", "records": n_rec, "compressed_bytes": C_bytes, "inflated_bytes": D_bytes,
        "zlib_level": wl["level"], "steps": args.steps, "warmup": args.warmup, "gpu": gpu_name_and_power(),
        "index_resident_ms_device": med([r[1] for r in res]), "index_resident_ms_wall": med([r[0] for r in res]),
        "index_resident_records_per_s": n_rec / (med([r[1] for r in res]) / 1e3),
        "index_e2e_ms_device": med([r[1] for r in ee]), "index_e2e_ms_wall": med([r[0] for r in ee]), "e2e_chunk_mb": args.chunk_mb,
        "index_e2e_records_per_s": n_rec / (med([r[0] for r in ee]) / 1e3),
        "index_stage_ms": {k: ix_stats[k] for k in ("ms_inflate", "ms_crc", "ms_scan", "ms_facets", "ms_total", "waves")},
        "qc_step_ms_device": med([r[1] for r in plain]), "qc_with_index_step_ms_device": med([r[1] for r in with_ix]),
        "qc_step_ms_wall": med([r[0] for r in plain]), "qc_with_index_step_ms_wall": med([r[0] for r in with_ix]),
        "index_extra_on_qc_step_pct_device": 100.0 * (med([r[1] for r in with_ix]) / med([r[1] for r in plain]) - 1.0),
        "bai_bytes": len(gpu_bai), "bai_chunks": chunks, "chunks_per_record": chunks / n_rec, "n_no_coor": parsed.n_no_coor,
        "bamgen_bai_bytes": int(bai_writer.size), "equal_to_bamgen_up_to_its_linear_clamp": bool(same_as_bamgen),
    }
    if not args.no_oracle:
        t = time.perf_counter()
        want_bytes = oracle_bai(pinned)
        out["oracle_single_thread_s"] = time.perf_counter() - t
        out["oracle_note"] = "single-thread restatement of the reference's `ngs index` loop over zlib (tests/cpp/bai_oracle.c), not the reference itself"
        out["equal_to_oracle"] = want_bytes == gpu_bai
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    lib.ngsq_host_free(pin)
    if not out["equal_to_bamgen_up_to_its_linear_clamp"] or out.get("equal_to_oracle") is False:
        raise SystemExit("the GPU index differs from the reference indexes")


def _index_run(eng_factory, flags, pinned, d_comp, C_bytes, blocks, n_blocks, pin=None, cuts=None):
    """One index-only run of a fresh engine: resident (d_comp) or streamed from pinned memory (cuts); (wall ms, device ms,
    engine)."""
    e = eng_factory(flags)
    t = time.perf_counter()
    if cuts is None:
        e.submit_device(d_comp.data_ptr(), C_bytes, blocks, n_blocks)
    else:
        for a, b in zip(cuts[:-1], cuts[1:]):
            if b == C_bytes:
                e.flush()
            e.submit_ptr(pin + a, b - a, a)
    e.finish()
    return (time.perf_counter() - t) * 1e3, e.stats()["ms_total"], e


def csi_bench(args, pinned, pin, blocks, n_blocks, n_rec, C_bytes, D_bytes, d_comp, cuts, wl, lib):
    import torch
    from ngs_b200 import ffi, formats
    from baiutil import oracle_bai
    from csiutil import oracle_csi
    med = lambda xs: float(np.median(xs))  # noqa: E731
    crc = ffi.NGSQ_F_VERIFY_CRC

    def factory(data, c_bytes, d_bytes, nb):
        def make(flags):
            e = ffi.Engine(flags=flags, reserve_compressed=c_bytes, reserve_inflated=d_bytes + 65536, reserve_blocks=nb + 16)
            hdr = formats.read_header(e, data)
            e.set_references([l for _, l in hdr.refs], [0] * len(hdr.refs))
            e.set_range(hdr.first_voffset, 0)
            return e
        return make

    make = factory(pinned, C_bytes, D_bytes, n_blocks)
    fmt = {"bai": ffi.NGSQ_F_INDEX | crc, "csi": ffi.NGSQ_F_INDEX | ffi.NGSQ_F_INDEX_CSI | crc}
    get = {"bai": lambda e: e.bai(), "csi": lambda e: e.csi()}
    res, ee, payload = {"bai": [], "csi": []}, {"bai": [], "csi": []}, {}
    for step in range(args.warmup + args.steps):
        for f in ("bai", "csi"):  # alternated
            w, d, e = _index_run(make, fmt[f], pinned, d_comp, C_bytes, blocks, n_blocks)
            payload.setdefault(f, get[f](e))
            assert get[f](e) == payload[f]
            e.close()
            if step >= args.warmup:
                res[f].append((w, d))
    for step in range(1 + args.steps):
        for f in ("bai", "csi"):
            w, d, e = _index_run(make, fmt[f], pinned, d_comp, C_bytes, blocks, n_blocks, pin=pin, cuts=cuts)
            assert get[f](e) == payload[f]
            e.close()
            if step:
                ee[f].append((w, d))
    # host assembly: the join of one part engine (the whole file) per format
    join = {"bai": ffi.join_bai, "csi": ffi.join_csi}
    assembly = {}
    for f in ("bai", "csi"):
        _, _, p = _index_run(make, (fmt[f] & ~ffi.NGSQ_F_INDEX) | ffi.NGSQ_F_INDEX_PART, pinned, d_comp, C_bytes, blocks, n_blocks)
        ts = []
        for _ in range(args.steps):
            t = time.perf_counter()
            assert join[f]([p]) == payload[f]
            ts.append((time.perf_counter() - t) * 1e3)
        assembly[f] = med(ts)
        p.close()
    csi = formats.parse_csi(payload["csi"])
    out = {
        "metric": "CSI (min_shift 14) against BAI build, index only", "records": n_rec, "compressed_bytes": C_bytes,
        "inflated_bytes": D_bytes, "zlib_level": wl["level"], "steps": args.steps, "warmup": args.warmup, "gpu": gpu_name_and_power(),
        "gpu_count": torch.cuda.device_count(), "csi_min_shift": csi.min_shift, "csi_depth": csi.depth,
    }
    for f in ("bai", "csi"):
        out[f"{f}_resident_ms_device"] = med([r[1] for r in res[f]])
        out[f"{f}_resident_ms_wall"] = med([r[0] for r in res[f]])
        out[f"{f}_e2e_ms_device"] = med([r[1] for r in ee[f]])
        out[f"{f}_e2e_ms_wall"] = med([r[0] for r in ee[f]])
        out[f"{f}_host_assembly_ms"] = assembly[f]
        out[f"{f}_bytes"] = len(payload[f])
    if not args.no_oracle:
        out["bai_equal_to_oracle"] = oracle_bai(pinned) == payload["bai"]
        out["csi_equal_to_oracle"] = oracle_csi(pinned) == payload["csi"]
    del d_comp
    torch.cuda.synchronize()
    lib.ngsq_host_free(pin)

    # shape 4: references past 2^29 and 2^30
    t0 = time.perf_counter()
    bam4, _, info4 = ffi.synth_bam(4, args.shape4_records, level=wl["level"])
    gen_s = time.perf_counter() - t0
    C4, D4 = int(bam4.size), int(info4["inflated_bytes"])
    b4, nb4, _ = ffi.bgzf_walk(bam4)
    d4 = torch.empty(C4 + 512, dtype=torch.uint8, device="cuda")
    d4[:C4].copy_(torch.from_numpy(np.asarray(bam4)))
    torch.cuda.synchronize()
    make4 = factory(bam4, C4, D4, nb4)
    r4, first = [], None
    for step in range(args.warmup + args.steps):
        w, d, e = _index_run(make4, fmt["csi"], bam4, d4, C4, b4, nb4)
        first = first or e.csi()
        assert e.csi() == first
        e.close()
        if step >= args.warmup:
            r4.append((w, d))
    _, _, p = _index_run(make4, ffi.NGSQ_F_INDEX_PART | ffi.NGSQ_F_INDEX_CSI | crc, bam4, d4, C4, b4, nb4)
    t = time.perf_counter()
    assert ffi.join_csi([p]) == first
    out["shape4"] = {"records": int(info4["n_records"]), "compressed_bytes": C4, "inflated_bytes": D4, "generate_s": gen_s,
                     "csi_depth": formats.parse_csi(first).depth, "csi_resident_ms_device": med([r[1] for r in r4]),
                     "csi_resident_ms_wall": med([r[0] for r in r4]), "csi_host_assembly_ms": (time.perf_counter() - t) * 1e3,
                     "csi_bytes": len(first)}
    if not args.no_oracle:
        out["shape4"]["csi_equal_to_oracle"] = oracle_csi(bam4) == first
    _emit(args, out)
    if out.get("csi_equal_to_oracle") is False or out.get("bai_equal_to_oracle") is False or out["shape4"].get("csi_equal_to_oracle") is False:
        raise SystemExit("the GPU index differs from the oracle's")


def _emit(args, out):
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


def parts_bench(args, pinned, pin, blocks, n_blocks, n_rec, C_bytes, D_bytes, d_comp_0, lib):
    import threading

    import torch
    from ngs_b200 import ffi, formats
    from baiutil import oracle_bai
    n = args.gpus
    if torch.cuda.device_count() < n:
        raise SystemExit(f"--gpus {n}: only {torch.cuda.device_count()} device(s) visible")
    crc = ffi.NGSQ_F_VERIFY_CRC
    starts = [blocks[i].coffset for i in range(n_blocks)]
    whole = ffi.Engine(0, flags=ffi.NGSQ_F_INDEX | crc, reserve_compressed=C_bytes, reserve_inflated=D_bytes + 65536, reserve_blocks=n_blocks + 16)
    hdr = formats.read_header(whole, pinned)
    lens = [l for _, l in hdr.refs]
    whole.set_references(lens, [0] * len(lens))
    whole.set_range(hdr.first_voffset, 0)
    whole.submit_device(d_comp_0.data_ptr(), C_bytes, blocks, n_blocks)
    whole.finish()
    one_bai = whole.bai()
    whole.close()
    # cuts by the driver's rule
    t = time.perf_counter()
    finder = ffi.Engine(0, flags=ffi.NGSQ_F_INDEX_PART)
    finder.set_references(lens, [0] * len(lens))
    base = hdr.first_voffset >> 16
    bounds = [hdr.first_voffset]
    for k in range(1, n):
        target = base + (C_bytes - base) * k // n
        i = int(np.searchsorted(np.asarray(starts, dtype=np.uint64), target))
        nb = 4
        v = 0
        while i < n_blocks and nb <= 4096:
            j = min(n_blocks, i + nb)
            hi = blocks[j - 1].coffset + blocks[j - 1].csize
            v, _ = finder.find_record(np.ascontiguousarray(pinned[starts[i]:hi]), starts[i])
            if v or j == n_blocks:
                break
            nb *= 2
        if v and v > bounds[-1]:
            bounds.append(v)
    finder.close()
    plan_ms = (time.perf_counter() - t) * 1e3
    ranges = []
    for k, first in enumerate(bounds):
        end = bounds[k + 1] if k + 1 < len(bounds) else 0
        lo, hi = formats.shard_byte_range(formats.Shard(first, end, []), blocks, n_blocks, C_bytes)
        ranges.append((first, end, lo, hi))
    del d_comp_0
    torch.cuda.empty_cache()
    engines, dev = [], []
    for k, (first, end, lo, hi) in enumerate(ranges):
        b0 = int(np.searchsorted(np.asarray(starts, dtype=np.uint64), lo))
        b1 = int(np.searchsorted(np.asarray(starts, dtype=np.uint64), hi)) if hi < C_bytes else n_blocks
        with torch.cuda.device(k):
            d = torch.empty(hi - lo + 512, dtype=torch.uint8, device=f"cuda:{k}")
            d[: hi - lo].copy_(torch.from_numpy(pinned[lo:hi]))
        sub = (ffi.Block * (b1 - b0))(*[blocks[i] for i in range(b0, b1)])
        e = ffi.Engine(k, flags=ffi.NGSQ_F_INDEX_PART | crc, reserve_compressed=hi - lo, reserve_inflated=D_bytes // len(ranges) * 2 + 65536,
                       reserve_blocks=b1 - b0 + 16)
        e.set_references(lens, [0] * len(lens))
        engines.append(e)
        dev.append((d, sub, b1 - b0))
    torch.cuda.synchronize()

    def step(mode):
        times = [None] * len(engines)

        def run(k):
            e, (first, end, lo, hi), (d, sub, nb) = engines[k], ranges[k], dev[k]
            t0 = time.perf_counter()
            e.reset()
            e.set_range(first, end)
            if mode == "resident":
                e.submit_device(d.data_ptr(), hi - lo, sub, nb)
            else:
                a = lo
                while a < hi:
                    b = min(hi, a + (args.chunk_mb << 20))
                    if b < hi:  # whole blocks per chunk
                        b = int(starts_np[int(np.searchsorted(starts_np, b))])
                    e.submit_ptr(pin + a, b - a, a)
                    a = b
            e.finish()
            times[k] = ((time.perf_counter() - t0) * 1e3, e.stats()["ms_total"])
        ts = [threading.Thread(target=run, args=(k,)) for k in range(len(engines))]
        t0 = time.perf_counter()
        for x in ts:
            x.start()
        for x in ts:
            x.join()
        wall = (time.perf_counter() - t0) * 1e3
        t1 = time.perf_counter()
        bai = ffi.join_bai(engines)
        join_ms = (time.perf_counter() - t1) * 1e3
        return wall, max(tt[1] for tt in times), join_ms, bai

    starts_np = np.asarray(starts, dtype=np.int64)
    for _ in range(args.warmup):
        step("resident")
    res = [step("resident") for _ in range(args.steps)]
    for _ in range(max(1, args.warmup // 2)):
        step("e2e")
    ee = [step("e2e") for _ in range(args.steps)]
    joined = res[-1][3]
    assert all(r[3] == joined for r in res + ee)
    med = lambda xs: float(np.median(xs))  # noqa: E731
    out = {
        "metric": "BAI build of a file without an index cut between devices (NGSQ_F_INDEX_PART + ngsq_join_bai)", "gpus": n,
        "parts": len(ranges), "records": n_rec, "compressed_bytes": C_bytes, "steps": args.steps, "warmup": args.warmup, "gpu": gpu_name_and_power(),
        "plan_ms_host": plan_ms,
        "index_resident_ms_device_slowest_part": med([r[1] for r in res]), "index_resident_ms_wall_parts": med([r[0] for r in res]),
        "index_e2e_ms_device_slowest_part": med([r[1] for r in ee]), "index_e2e_ms_wall_parts": med([r[0] for r in ee]), "e2e_chunk_mb": args.chunk_mb,
        "join_ms_host": med([r[2] for r in res + ee]),
        "index_resident_ms_wall_with_join": med([r[0] + r[2] for r in res]),
        "index_e2e_ms_wall_with_join": med([r[0] + r[2] for r in ee]),
        "equal_to_one_engine": joined == one_bai, "bai_bytes": len(joined),
    }
    if not args.no_oracle:
        out["equal_to_oracle"] = oracle_bai(pinned) == joined
    _emit(args, out)
    for e in engines:
        e.close()
    lib.ngsq_host_free(pin)
    if not out["equal_to_one_engine"] or out.get("equal_to_oracle") is False:
        raise SystemExit("the joined index differs from one engine's or the oracle's")


def driver_bench(args, bam, bai_writer, n_rec):
    import shutil
    import tempfile
    from baiutil import oracle_bai  # noqa: F401
    drv = os.path.join(ROOT, "ngs_b200", "ngs-cuda-qc")
    d = tempfile.mkdtemp(prefix="index_bench_")
    try:
        src = os.path.join(d, "w.bam")
        bam.tofile(src)
        del bam

        def run(cmd):
            r = subprocess.run([drv] + cmd, capture_output=True, text=True)
            if r.returncode:
                raise SystemExit(r.stderr)

        def two():
            os.remove(src + ".bai") if os.path.exists(src + ".bai") else None
            t = time.perf_counter()
            run(["index", src])
            run(["qc", src, "GRCh38_no_alt_AnalysisSet", "-o", d, "-p", "two"])
            return (time.perf_counter() - t) * 1e3

        def one():
            os.remove(src + ".bai") if os.path.exists(src + ".bai") else None
            t = time.perf_counter()
            run(["qc", src, "GRCh38_no_alt_AnalysisSet", "-o", d, "-p", "one", "--cuda-build-index"])
            return (time.perf_counter() - t) * 1e3

        for _ in range(args.warmup):
            two()
            one()
        a, b = [], []
        for _ in range(args.steps):  # alternated
            a.append(two())
            b.append(one())
        same = open(os.path.join(d, "one.results.json")).read() == open(os.path.join(d, "two.results.json")).read()
        med = lambda xs: float(np.median(xs))  # noqa: E731
        out = {"metric": "host driver wall time from a file, qc --cuda-build-index vs index + qc", "records": n_rec, "steps": args.steps,
               "gpu": gpu_name_and_power(), "io": "O_DIRECT reads (the page cache does not serve the BAM)",
               "index_then_qc_ms_wall": med(a), "qc_build_index_ms_wall": med(b), "all_index_then_qc_ms": a, "all_qc_build_index_ms": b,
               "same_results_json": same}
        _emit(args, out)
    finally:
        shutil.rmtree(d, ignore_errors=True)


if __name__ == "__main__":
    main()
