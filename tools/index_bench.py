"""Measures the GPU BAI build (NGSQ_F_INDEX) on bench.py's default workload: the same 2x150bp WGS-shaped synthetic BAM (bench
seed, shape and zlib level; 100 M records unless --records), indexed

  * resident: the compressed file in HBM, ngsq_submit_device + ngsq_finish + ngsq_get_bai, index only;
  * end to end: ngsq_submit from pinned host memory in --chunk-mb chunks, index only;
  * beside qc: bench.py's resident qc step (record facets + coverage + CRC) with and without NGSQ_F_INDEX, alternated.

Device times are the engine's CUDA-event totals (ms_total); wall times are host clocks around calls that end in a device
synchronise and include the host's assembly of the .bai.  The result is compared with the oracle's single-thread index of
the same file (tests/cpp/bai_oracle.c, a restatement of the reference's `ngs index` loop over zlib; its time is the CPU
baseline) and with bamgen's (equal up to bamgen's clamped linear index).  Prints one JSON line; --out writes it too.

  python tools/index_bench.py [--records N] [--steps K] [--warmup W] [--chunk-mb M] [--no-oracle] [--out FILE]
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


if __name__ == "__main__":
    main()
