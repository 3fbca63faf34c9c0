#!/usr/bin/env python
"""bench.py — `ngs qc` BAM hot path on B200 (BASELINE.json metric: records/s and decompressed GB/s).

A "step" is one full pass of the hot path over one synthetic BAM shard per GPU, streamed in waves:
BGZF inflate -> CRC -> record scan -> record facets + coverage scatter (per wave) -> coverage resolve (-> NCCL merge).

  value   device-timed (CUDA events on the engine's stream, max over ranks), compressed BAM
          already resident in HBM when the timed region starts.
  e2e     the same pass through the host-facing C ABI (ngsq_submit from pinned HOST memory in
          chunks, results read back to the host), H2D/D2H inside the timed region, wall clock
          bracketed by barrier + device synchronize.
  parity  the TIMED runs' own result buffers (last resident step and last e2e step, after the NCCL merge at N>1)
          are compared with the committed full-size golden of the workload (tests/golden/fullsize_*.npz: the
          oracle's integers over exactly these shard files); a difference fails the run.
  --dump-outputs DIR   the last timed resident step's results (every integer array the C ABI returns, as float64)
          go to DIR/<name>.npy.  The synthetic inputs are seeded, so two builds run with the same arguments can be
          compared file for file.
  --impl reference   the CPU oracle (restatement of the reference's single-threaded algorithm;
          the Rust reference cannot be built in this image) on a bounded sample, rank 0 only.

Workloads (--shape): wgs (default) N=1 -> configs[1] (100M-record 2x150 WGS BAM, all facets incl. coverage);
N>1 -> one logical 75M*N-record BAM (N=8: configs[2], 600M records) partitioned by contig ranges (LPT over
record counts); every rank generates exactly its shard, results merged by one NCCL all-reduce.
c1 / c4 / c5 -> configs[0] / [3] / [4] (profiles/ holds their lines; the driver's default run is wgs).
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def parse_args():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=3)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--shape", default="wgs", choices=sorted(WORKLOADS), help="workload (BASELINE.json configs): wgs = configs[1]/[2], c1, c4, c5")
    p.add_argument("--records", type=int, default=0, help="records per GPU (default: the named config's size)")
    p.add_argument("--level", type=int, default=-1, help="zlib level of the synthetic BAM (default 1 for >=20M records, else 6)")
    p.add_argument("--chunk-mb", type=int, default=256, help="e2e submit chunk size")
    p.add_argument("--cpu-sample", type=int, default=3_000_000, help="records in the CPU-baseline sample")
    p.add_argument("--no-crc", action="store_true", help="skip the per-block CRC32 check (reference verifies it)")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-cpu", action="store_true")
    p.add_argument("--dump-outputs", metavar="DIR", default=None,
                   help="write the results of the last timed device-resident step to DIR/<name>.npy (float64)")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    return args


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (profiling guide recipe)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        # median over samples under load (top half of the observed clocks)
        sm_sorted = sorted(sm)
        under_load = sm_sorted[len(sm_sorted) // 2:] if sm_sorted else []
        return {"sm_mhz": float(np.median(under_load)) if under_load else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


GC_SEED = 7

# name -> (generator shape, records per GPU at N=1, records per GPU at N>1, record facets, coverage)
# BASELINE.json configs: wgs = configs[1] (N=1, 100 M) / configs[2] (N=8: 600 M = 75 M per GPU); c1 = configs[0];
# c4 = configs[3] (long reads); c5 = configs[4] (RNA-seq)
WORKLOADS = {
    "wgs": (1, 100_000_000, 75_000_000, True, True),
    "c1": (0, 1_000_000, 1_000_000, True, False),
    "c4": (2, 2_000_000, 2_000_000, True, True),
    "c5": (3, 200_000_000, 200_000_000, True, True),
}
WORKLOAD_TEXT = {
    "wgs": "2x150bp WGS-shaped synthetic BAM, all facets incl. coverage",
    "c1": "2x150bp coordinate-sorted synthetic BAM over a 3-contig reference, record-based facets only",
    "c4": "long-read (10-50 kb, dense CIGARs) synthetic BAM, all facets incl. coverage",
    "c5": "spliced 2x100bp RNA-seq-shaped synthetic BAM (CIGAR N skips, high duplicate/secondary rates), all facets incl. coverage",
}


def workload(name, n_ranks, per_gpu=0, level=-1):
    """The bench workload `name` at n_ranks GPUs: one logical BAM of per_gpu * n_ranks records, cut into
    contig-exclusive shards (LPT by record count).  Deterministic: tests/golden/make_fullsize_goldens.py builds the
    goldens from the same description."""
    from ngs_b200 import ffi
    shape, one, many, records, coverage = WORKLOADS[name]
    per_gpu = per_gpu or (one if n_ranks == 1 else many)
    total = per_gpu * n_ranks
    if level < 0:
        # zlib level 1 bounds the generation time of the multi-GB workloads (DESIGN.md section 6); long reads: 56 KB per record
        level = 1 if per_gpu >= 20_000_000 or shape == 2 else 6
    per_contig, tail = ffi.synth_layout(shape, total)
    parts, loads = lpt_partition(per_contig, n_ranks)
    return {"name": name, "shape": shape, "n_ranks": n_ranks, "per_gpu": per_gpu, "total_records": total, "level": level,
            "records": records, "coverage": coverage, "parts": parts, "tail_rank": int(np.argmin(loads)),
            "key": f"{name}_n{n_ranks}_{total}_l{level}"}


def workload_shard(wl, rank):
    """(contig mask, with_tail) of the shard file rank `rank` generates."""
    return sum(1 << c for c in wl["parts"][rank]), rank == wl["tail_rank"]


def lpt_partition(weights, n_parts):
    """Longest-processing-time packing of contigs onto shards (contig-exclusive ownership)."""
    order = sorted(range(len(weights)), key=lambda c: -weights[c])
    loads = [0] * n_parts
    parts = [[] for _ in range(n_parts)]
    for c in order:
        k = min(range(n_parts), key=lambda i: loads[i])
        parts[k].append(c)
        loads[k] += weights[c]
    return parts, loads


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(res, out_dir):
    """Writes the integer results a caller of the engine receives (helpers.collect) as float64 .npy files, so that two
    builds can be compared output for output.  Every count is below 2**53, so float64 holds it exactly."""
    arrays = {}
    if "general" in res:
        arrays.update(general=res["general"], tlen_hist=res["tlen_hist"], tlen_counts=[res["tlen_processed"], res["tlen_ignored"]],
                      gc_hist=res["gc_hist"], gc_nuc=res["gc_nuc"], gc_rec=res["gc_rec"], quality=res["quality"])
    if "coverage" in res:
        contigs = sorted(res["coverage"])
        cov = [res["coverage"][c] for c in contigs]
        arrays.update(coverage_contigs=contigs, coverage_hist=np.array([v["hist"] for v in cov], dtype=np.uint64).reshape(len(cov), 2049),
                      coverage_too_large=[v["too_large"] for v in cov], coverage_n_bins=[len(v["bin_sums"]) for v in cov],
                      coverage_bin_sums=np.concatenate([v["bin_sums"] for v in cov]) if cov else [],
                      nonsensical=[res["nonsensical"]])
    arrays = {k: np.asarray(v, dtype=np.uint64) for k, v in arrays.items()}
    for k, a in arrays.items():
        if a.size and int(a.max()) >= 1 << 53:
            raise SystemExit(f"--dump-outputs: {k} holds a count that float64 cannot represent exactly")
    total = sum(8 * a.size for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes of results exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, f"{k}.npy"), a.astype(np.float64))


def cpu_sample(args, wl):
    """Bounded CPU sample that keeps the workload's SHAPE: whole contigs of the N=1 logical BAM of the shape at full
    depth (so the per-record and the per-position costs of the reference keep their proportion — a shallow
    whole-genome sample would charge the reference its 3.1 Gbp coverage sweep for 3 % of the records).  Contigs are
    taken from the small end until about --cpu-sample records are reached.  The same sample at every N.
    Long reads (56 KB per record, 340 k records on the smallest contig) cannot be sampled by whole contigs: there the
    sample is a smaller logical BAM of the same shape, sized for the same number of BASES."""
    from ngs_b200 import ffi
    shape, total, level = wl["shape"], wl["per_gpu"], wl["level"]
    if shape == 3:
        # spliced reads: the reference's Coverage.process is O(span) and 60 % of these records span a ~100 kb intron
        # (coverage.rs:165-178 walks every skipped position): 3 M records would be minutes of one core
        # (measured: 101 s for the smallest chromosome of the 200 M-record BAM).  Whole contigs of a logical BAM at a quarter
        # of the depth instead: the smallest chromosome then holds ~750 k records
        args = argparse.Namespace(**{**vars(args), "cpu_sample": min(args.cpu_sample, 800_000)})
        total = max(total // 4, 1_000_000)
    if shape == 2:
        n = max(2000, min(total, args.cpu_sample * 300 // 56000))
        bam, bai, info = ffi.synth_bam(shape, n, level=level)
        return bam, bai, info, f"{info['n_records']} records of the same long-read shape over the same 5 contigs (zlib-{level})"
    per_contig, _ = ffi.synth_layout(shape, total)
    order = sorted(range(len(per_contig)), key=lambda c: per_contig[c])
    mask, n = 0, 0
    for c in order:
        if per_contig[c] == 0:
            continue
        if n >= args.cpu_sample:
            break
        # once past half the target, do not overshoot it by more than half (the first real contig is always taken)
        if n > args.cpu_sample * 0.5 and n + per_contig[c] > args.cpu_sample * 1.5:
            break
        mask |= 1 << c
        n += per_contig[c]
    bam, bai, info = ffi.synth_bam(shape, total, level=level, contig_mask=mask, with_tail=False)
    contigs = [c for c in range(len(per_contig)) if mask >> c & 1]
    desc = (f"{info['n_records']} records = contigs {contigs} of the {total}-record {wl['name']}-shaped BAM at full depth "
            f"(zlib-{level})")
    return bam, bai, info, desc


def run_reference(args, rank, emit):
    """CPU arm: oracle (port of the reference algorithm, 1 thread like the reference) on a bounded sample."""
    if rank != 0:
        return
    from helpers import oracle_ints
    wl1 = workload(args.shape, 1, args.records, args.level)
    bam, bai, info, desc = cpu_sample(args, wl1)
    n = info["n_records"]
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        oracle_ints(bam, bai, gc_seed=GC_SEED, records=wl1["records"], coverage=wl1["coverage"])
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
        if sum(times) > 150:  # bounded: never let the CPU arm run away
            break
    per = float(np.mean(times))
    val = n / per
    passes = int(wl1["records"]) + int(wl1["coverage"])
    line = {
        "impl": "reference", "metric": "ngs qc records/sec", "value": val, "unit": "records/s", "n_gpus": args.gpus,
        "steps": len(times), "warmup": args.warmup, "ms_per_step": per * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/u64", "data": "synthetic",
        "decompressed_gbs": info["inflated_bytes"] * passes / per / 1e9,
        "config": {"workload": f"{WORKLOAD_TEXT[args.shape]} (bounded sample of the named config: {desc})",
                   "sample_records": n, "note": "CPU restatement of the reference (oracle/ngsqc_oracle.c, zlib inflate, one pass per facet family, 1 thread: the reference's qc path is single-threaded); the Rust reference cannot be built in this image"},
        "cpu_baseline": {"value": val, "unit": "records/s", "cores": 1, "kind": "port", "sample": desc + f", {passes} pass(es)"},
        "e2e": {"value": val, "unit": "records/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


_T0 = time.perf_counter()


def log(msg):
    """Progress on stderr (stdout carries only the JSON line): makes a hang on a GPU box diagnosable."""
    print(f"[bench r{os.environ.get('RANK', '0')} +{time.perf_counter() - _T0:7.1f}s] {msg}", file=sys.stderr, flush=True)


def bind_to_gpu_numa_node(local_rank):
    """Pins this process to the CPUs of the GPU's NUMA node before any pinned allocation (first touch decides where the
    staging memory lives).  Returns a short description for the JSON line."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(local_rank)], capture_output=True, text=True).stdout.strip()
        bdf = out.lower().replace("00000000:", "0000:") if out else None
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read()) if bdf else -1
        if node < 0:
            return {"numa_node": node, "bound": False}
        cpus = open(f"/sys/devices/system/node/node{node}/cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            a, _, b = part.partition("-")
            ids.update(range(int(a), int(b or a) + 1))
        os.sched_setaffinity(0, ids & os.sched_getaffinity(0) or os.sched_getaffinity(0))
        return {"numa_node": node, "bound": True, "cpus": cpus}
    except Exception as ex:  # never fail the bench over a binding
        return {"numa_node": None, "bound": False, "error": str(ex)[:80]}


def main():
    args = parse_args()
    # stdout carries exactly ONE JSON line: libraries that print there (NCCL prints its version banner on
    # stdout) are redirected to stderr, the line is written to the saved descriptor
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        os.write(json_fd, (json.dumps(line) + "\n").encode())

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, emit)
        return
    if world != args.gpus and world > 1:
        args.gpus = world

    import torch
    import torch.distributed as dist
    from ngs_b200 import ffi, formats
    from helpers import assert_same_ints, collect, compare_fullsize, engine_ints, oracle_ints

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the ngs-cuda engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    N = args.gpus
    numa = bind_to_gpu_numa_node(local_rank)
    if N > 1:
        log("init_process_group")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if N > 1:
            dist.barrier()
        torch.cuda.synchronize()

    wl = workload(args.shape, N, args.records, args.level)
    shape, level, total_records = wl["shape"], wl["level"], wl["total_records"]
    named = args.records == 0 and args.level < 0  # the size BASELINE.json names for this shape

    # ---- this rank's shard of the logical BAM (contig-exclusive, LPT by record count) ----
    mask, with_tail = workload_shard(wl, rank)
    t0 = time.perf_counter()
    bam, bai, info = ffi.synth_bam(shape, total_records, level=level, contig_mask=mask, with_tail=with_tail)
    gen_s = time.perf_counter() - t0
    log(f"generated shard: {info['n_records']} records, {bam.size} bytes in {gen_s:.1f}s")
    n_rec = info["n_records"]
    C_bytes, D_bytes = int(bam.size), int(info["inflated_bytes"])

    # pinned host copy (e2e source) and device-resident copy (value source)
    lib = ffi.load_library()
    pin_ptr = lib.ngsq_host_alloc(C_bytes)
    if not pin_ptr:
        raise SystemExit("cudaHostAlloc failed")
    pinned = np.ctypeslib.as_array(C.cast(pin_ptr, C.POINTER(C.c_uint8)), shape=(C_bytes,))
    pinned[:] = bam
    del bam
    blocks, n_blocks, used = ffi.bgzf_walk(pinned)
    assert used == C_bytes
    flags = ((ffi.NGSQ_F_RECORD_FACETS if wl["records"] else 0) | (ffi.NGSQ_F_COVERAGE if wl["coverage"] else 0)
             | (0 if args.no_crc else ffi.NGSQ_F_VERIFY_CRC))
    # the engine streams: two wave slots of inflated bytes whatever the file size; the compressed shard stays resident
    # here because the device-timed `value` needs it in HBM when the timed region starts
    eng = ffi.Engine(device=local_rank, flags=flags, gc_seed=GC_SEED, reserve_compressed=C_bytes, reserve_inflated=D_bytes + 65536,
                     reserve_blocks=n_blocks + 16)
    hdr = formats.read_header(eng, pinned)
    names = [n for n, _ in hdr.refs]
    lens = [l for _, l in hdr.refs]
    # the same coverage mask on every rank: the packed result layout (the NCCL payload) depends on it;
    # contigs a rank does not own stay untouched there and contribute zeros to the reduce
    enabled = [1 if formats.is_primary(nm) else 0 for nm in names]
    eng.set_references(lens, enabled)
    eng.set_range(hdr.first_voffset, 0)
    d_comp = torch.empty(C_bytes + 512, dtype=torch.uint8, device=dev)
    d_comp[:C_bytes].copy_(torch.from_numpy(pinned))
    torch.cuda.synchronize()

    log("engine ready, compressed shard resident")
    if N > 1:
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid.copy_(torch.frombuffer(bytearray(ffi.nccl_unique_id()), dtype=torch.uint8))
        dist.broadcast(uid, 0)
        eng.comm_init(N, rank, bytes(uid.cpu().numpy().tobytes()))
        log("engine NCCL communicator ready")

    def step_resident():
        eng.reset()
        eng.submit_device(d_comp.data_ptr(), C_bytes, blocks, n_blocks)
        eng.finish()
        if N > 1:
            eng.reduce(0)
        return eng.stats()

    chunk = args.chunk_mb << 20
    # chunk boundaries on whole blocks (host-side K1 framing, done once: it is I/O bookkeeping)
    cuts = [0]
    acc = 0
    for i in range(n_blocks):
        acc += blocks[i].csize
        if acc - cuts[-1] >= chunk:
            cuts.append(acc)
    if cuts[-1] != C_bytes:
        cuts.append(C_bytes)

    def step_e2e():
        eng.reset()
        for a, b in zip(cuts[:-1], cuts[1:]):
            eng.submit_ptr(pin_ptr + a, b - a, a)
        eng.finish()
        if N > 1:
            eng.reduce(0)
        return collect(eng, lens, enabled, wl["records"], wl["coverage"])  # D2H of every result the host consumes

    # ---- warm-up ----
    for i in range(max(args.warmup, 3)):
        st = step_resident()
        log(f"warm-up {i}: {st['ms_total']:.1f} ms")
    # ---- timed: device-resident ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    t0 = time.perf_counter()
    dev_ms, red_ms, tot_ms, infl_ms, dec_ms_l, res_ms_l, stats = [], [], [], [], [], [], None
    for _ in range(args.steps):
        stats = step_resident()
        dev_ms.append(stats["ms_total"] + stats["ms_reduce"])
        red_ms.append(stats["ms_reduce"])
        tot_ms.append(stats["ms_total"])
        infl_ms.append(stats["ms_inflate"])
        dec_ms_l.append(stats["ms_inflate_decode"])
        res_ms_l.append(stats["ms_inflate_resolve"])
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3 / args.steps
    clocks = sampler.stop()
    dev_step_ms = float(np.mean(dev_ms))
    res_resident = collect(eng, lens, enabled, wl["records"], wl["coverage"])  # the last TIMED step's own results
    if args.dump_outputs and rank == 0:  # after the NCCL merge, rank 0 holds the results of the whole logical BAM
        dump_outputs(res_resident, args.dump_outputs)

    # ---- timed: end to end from pinned host memory ----
    log(f"resident steps done: {dev_step_ms:.1f} ms/step")
    e2e_ms = None
    res_e2e = None
    e2e_tail = None
    h2d_gbs = None
    if not args.no_e2e:
        step_e2e()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res_e2e = step_e2e()
        barrier()
        e2e_ms = (time.perf_counter() - t0) * 1e3 / args.steps
        e2e_tail = res_e2e["stats"]["ms_tail"]
        # the box's host-to-device ceiling with all ranks copying at once: the same pinned buffer, the same chunks,
        # no kernels — what an e2e step could reach if the GPU work were free
        scratch = torch.empty(min(C_bytes, 4 << 30) + 512, dtype=torch.uint8, device=dev)
        src = torch.from_numpy(pinned[: scratch.numel() - 512])
        scratch[: src.numel()].copy_(src, non_blocking=True)
        barrier()
        t0 = time.perf_counter()
        for _ in range(2):
            scratch[: src.numel()].copy_(src, non_blocking=True)
        barrier()
        h2d_gbs = 2 * src.numel() / (time.perf_counter() - t0) / 1e9
        del scratch

    log("e2e steps done")
    # ---- the kernels' own times: one more resident pass with every kernel of a wave on ONE stream (NGSQ_F_SERIAL_STAGES).
    # In the timed steps the scan / facet / CRC kernels of wave k share the SMs with the inflate of wave k+1, so the per-stage
    # event times there include each other; this pass is NOT part of `value`.
    serial = None
    if N == 1:
        eng_s = ffi.Engine(device=local_rank, flags=flags | ffi.NGSQ_F_SERIAL_STAGES, gc_seed=GC_SEED, reserve_inflated=D_bytes + 65536,
                           reserve_blocks=n_blocks + 16)
        eng_s.set_references(lens, enabled)
        eng_s.set_range(hdr.first_voffset, 0)
        for _ in range(2):
            eng_s.reset()
            eng_s.submit_device(d_comp.data_ptr(), C_bytes, blocks, n_blocks)
            eng_s.finish()
        ss = eng_s.stats()
        same = "identical"
        try:
            assert_same_ints(collect(eng_s, lens, enabled, wl["records"], wl["coverage"]), res_resident, records=wl["records"], coverage=wl["coverage"])
        except AssertionError as ex:
            same = "DIFFERENT: " + " ".join(str(ex).split())[:200]
        serial = {"ms_per_step": ss["ms_total"], "results_vs_timed_run": same,
                  "stage_ms": {k: ss[k] for k in ["ms_inflate", "ms_inflate_decode", "ms_inflate_resolve", "ms_crc", "ms_scan", "ms_facets", "ms_coverage"]},
                  "decode_launch_ms": ss["ms_inflate_decode"] / max(ss["inflate_launches"], 1)}
        eng_s.close()
        log(f"serial-stages pass: {ss['ms_total']:.1f} ms")
    # ---- max over ranks ----
    agg = torch.tensor([dev_step_ms, wall_ms, e2e_ms or 0.0, float(np.mean(infl_ms)), float(np.mean(tot_ms)), -float(np.mean(tot_ms)),
                        float(np.mean(red_ms)), -(h2d_gbs or 0.0), e2e_tail or 0.0], dtype=torch.float64, device=dev)
    tot = torch.tensor([n_rec, C_bytes, D_bytes, stats["records"], (res_e2e or res_resident)["stats"]["records"]], dtype=torch.float64, device=dev)
    if N > 1:
        dist.all_reduce(agg, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    dev_step_ms, wall_ms, e2e_ms_max, infl_ms_max, tot_ms_max, neg_tot_ms_min, red_ms_max, neg_h2d_min, e2e_tail_max = [float(x) for x in agg.cpu()]
    all_rec, all_C, all_D, got_rec_resident, got_rec_e2e = [float(x) for x in tot.cpu()]

    # ---- parity of the TIMED runs against the committed full-size golden (rank 0 holds the merged integers) ----
    parity = None
    parity_failed = None
    if rank == 0:
        try:
            verdicts = []
            for label, res, got_rec in (("resident", res_resident, got_rec_resident), ("e2e", res_e2e, got_rec_e2e)):
                if res is None:
                    continue
                assert int(got_rec) == int(all_rec), f"{label}: engine counted {int(got_rec)} records, the generator wrote {int(all_rec)}"
                v = compare_fullsize(res, wl["key"], n_records=all_rec)
                verdicts.append((label, v))
            if verdicts and all(v for _, v in verdicts):
                parity = "timed " + " and ".join(l for l, _ in verdicts) + " runs: " + verdicts[0][1]
            else:
                parity = (f"record counts of the timed runs equal the generator's ({int(all_rec)}); no full-size golden committed for {wl['key']} "
                          "(sample parity below)")
        except AssertionError as ex:
            parity_failed = "FAILED: " + " ".join(str(ex).split())[:300]
            parity = parity_failed

    # ---- N-rank parity on ONE file: BAI-derived shards + the engine's NCCL merge vs the oracle's whole-file integers ----
    cpu = None
    sample_parity = None
    merged_parity = None
    if N > 1 and not args.no_cpu:
        sn = args.cpu_sample
        sb, sbai, _ = ffi.synth_bam(shape, sn, level=6)      # every rank writes the same bytes (deterministic generator)
        hdr_s = formats.read_header(eng, sb)
        sblocks, sn_blocks, _ = ffi.bgzf_walk(sb)
        shards = formats.plan_shards(hdr_s, formats.parse_bai(sbai.tobytes()), N, sb.size)
        sh = shards[rank]
        eng.reset()
        if sh.contigs:
            lo, hi = formats.shard_byte_range(sh, sblocks, sn_blocks, sb.size)
            eng.set_range(sh.first_voffset, sh.end_voffset)
            eng.submit(np.ascontiguousarray(sb[lo:hi]), lo)
        else:
            eng.set_range(0, 0)
        eng.finish()
        eng.reduce(0)
        if rank == 0:
            try:
                got_m = collect(eng, lens, enabled, wl["records"], wl["coverage"])
                assert_same_ints(got_m, oracle_ints(sb, sbai, gc_seed=GC_SEED, records=wl["records"], coverage=wl["coverage"]),
                                 records=wl["records"], coverage=wl["coverage"], gc_window=True)
                cut_inside = sum(1 for s in shards if s.end_voffset & 0xFFFF)
                merged_parity = (f"ONE {sn}-record file cut into {N} BAI-derived shards ({cut_inside} cuts inside a BGZF block), one shard per rank, "
                                 "engine NCCL merge: bit-exact vs the oracle on the whole file, GC window histogram included")
            except AssertionError as ex:  # never leave the other ranks waiting
                merged_parity = "FAILED: " + " ".join(str(ex).split())[:300]
        eng.reset()
        eng.set_range(hdr.first_voffset, 0)
        log("merged parity checked")
    if rank == 0 and not args.no_cpu:
        wl1 = workload(args.shape, 1, args.records, args.level)
        sbam, sbai, sinfo, sdesc = cpu_sample(args, wl1)
        sn = sinfo["n_records"]
        t0 = time.perf_counter()
        want = oracle_ints(sbam, sbai, gc_seed=GC_SEED, records=wl["records"], coverage=wl["coverage"])
        cpu_s = time.perf_counter() - t0
        got = engine_ints(sbam, gc_seed=GC_SEED, device=local_rank, records=wl["records"], coverage=wl["coverage"])
        try:
            assert_same_ints(got, want, records=wl["records"], coverage=wl["coverage"])
            sample_parity = "bit-exact vs oracle on the CPU-baseline sample (all integer outputs)"
        except AssertionError as ex:
            sample_parity = "FAILED: " + " ".join(str(ex).split())[:300]
        cpu = {"value": sn / cpu_s, "unit": "records/s", "cores": 1, "kind": "port",
               "sample": f"{sdesc}, {int(wl['records']) + int(wl['coverage'])} pass(es), {cpu_s:.1f} s; host has {os.cpu_count()} cores, the reference qc path uses 1"}

    if rank == 0:
        peak, peak_kind = measured_peak()
        launches = max(stats["inflate_launches"], 1)
        dec_ms = float(np.mean(dec_ms_l)) / launches   # average launch duration of the dominant kernel (CUDA events)
        res_ms = float(np.mean(res_ms_l)) / launches
        # algorithmic bytes of the decode kernel per launch: compressed bytes read + inflated bytes written
        # (every 16-byte chunk is written once: literals, in-place match tokens, zeros elsewhere)
        achieved = (C_bytes + D_bytes) / launches / (dec_ms * 1e-3) / 1e9 if dec_ms > 0 else 0.0
        traffic = None
        try:
            with open(os.path.join(ROOT, "profiles", "inflate_traffic.json")) as f:
                tj = json.load(f)
                # ncu dram bytes per launch are proportional to the workload: scale from the profiled size
                traffic = tj["decode_dram_bytes_per_inflated_byte"] * D_bytes / launches
        except Exception:
            pass
        cov_bytes = sum(8 * (L + 2) for c, L in enumerate(lens) if enabled[c]) if wl["coverage"] else 0
        A = all_C + 2 * all_D + cov_bytes
        config_name = {"wgs": "configs[1]" if N == 1 else ("configs[2]" if N == 8 else "configs[1]/[2] family"), "c1": "configs[0]", "c4": "configs[3]", "c5": "configs[4]"}[args.shape]
        line = {
            "metric": "ngs qc records/sec", "value": all_rec / (dev_step_ms * 1e-3), "unit": "records/s", "n_gpus": N,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": dev_step_ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8/u64", "data": "synthetic",
            "decompressed_gbs": all_D / (dev_step_ms * 1e-3) / 1e9,
            "pipeline_hbm_frac": A / (dev_step_ms * 1e-3) / 1e9 / (peak * N),
            "wall_ms_per_step": wall_ms,
            "config": {"workload": (f"{config_name}: {int(all_rec)}-record {WORKLOAD_TEXT[args.shape]}" if named else
                                    f"{int(all_rec)}-record {WORKLOAD_TEXT[args.shape]} (NOT the named size of {config_name})")
                                   + (f", partitioned by contig ranges over {N} GPUs ({wl['per_gpu']} records per GPU; N=1 runs configs[1] = 100 M per GPU)" if N > 1 else ""),
                       "records": int(all_rec), "compressed_bytes": int(all_C), "inflated_bytes": int(all_D), "zlib_level": level,
                       "crc_check": not args.no_crc, "waves_per_gpu": int(stats["waves"]),
                       "l2": "inputs (GBs) far exceed the 126 MB L2; no flush needed", "generation_s": gen_s,
                       "stage_ms": {k: stats[k] for k in ["ms_inflate", "ms_inflate_decode", "ms_inflate_resolve", "ms_crc", "ms_scan", "ms_facets", "ms_coverage", "ms_tail"]},
                       "stage_ms_note": "event times inside the timed steps: the scan, facet and CRC kernels of wave k run beside the inflate of wave k+1, so the "
                                        "stages overlap and their sum exceeds ms_per_step; `serial_stages` holds the kernels' own times (one extra pass, one stream)",
                       "serial_stages": serial,
                       "ms_reduce": red_ms_max, "rank_ms_total": {"max": tot_ms_max, "min": -neg_tot_ms_min},
                       "stage_gbs": {"inflate (C+D)/t": (C_bytes + D_bytes) / (stats["ms_inflate"] * 1e-3) / 1e9 if stats["ms_inflate"] else None,
                                     "resolve D/t": D_bytes / (res_ms * launches * 1e-3) / 1e9 if res_ms else None,
                                     "crc D/t": D_bytes / (stats["ms_crc"] * 1e-3) / 1e9 if stats["ms_crc"] else None,
                                     "scan+facets D/t": D_bytes / ((stats["ms_scan"] + stats["ms_facets"]) * 1e-3) / 1e9,
                                     "coverage 8*sum(L)/t": cov_bytes / (stats["ms_coverage"] * 1e-3) / 1e9 if stats["ms_coverage"] and cov_bytes else None}},
            "roofline": {"bound": "hbm", "kernel": "inflate_decode_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_kind": peak_kind,
                         "launch_ms": dec_ms, "launches_per_step": launches,
                         "alone": None if not serial or not serial["decode_launch_ms"] else {
                             "launch_ms": serial["decode_launch_ms"],
                             "achieved": (C_bytes + D_bytes) / launches / (serial["decode_launch_ms"] * 1e-3) / 1e9,
                             "frac": (C_bytes + D_bytes) / launches / (serial["decode_launch_ms"] * 1e-3) / 1e9 / peak,
                             "what": "the same kernel without co-runners (serial_stages pass); `achieved` above is inside the timed steps, where the previous "
                                     "wave's scan kernels share the SMs with it"},
                         "note": "algorithmic bytes = compressed read + inflated written per launch; Huffman decode is instruction-issue bound, not HBM-bound (DESIGN.md section 4)"},
            "cpu_baseline": cpu,
            "e2e": None if args.no_e2e else {"value": all_rec / (e2e_ms_max * 1e-3), "unit": "records/s", "h2d_bytes_per_step": int(all_C),
                                             "d2h_bytes_per_step": int(8 * (1216 + 94 * 256 + sum(2052 + L // 50000 + 2 for L in lens))), "ms_per_step": e2e_ms_max,
                                             "ms_tail_after_last_wave_starts": e2e_tail_max,
                                             "device_ms_total": res_e2e["stats"]["ms_total"], "waves": int(res_e2e["stats"]["waves"]),
                                             "stage_ms": {k: res_e2e["stats"][k] for k in ["ms_inflate", "ms_inflate_decode", "ms_inflate_resolve", "ms_crc", "ms_scan", "ms_facets", "ms_coverage"]},
                                             "h2d_ceiling_gbs_per_gpu": -neg_h2d_min,
                                             "h2d_ceiling_ms": (C_bytes / 1e9) / (-neg_h2d_min) * 1e3 if neg_h2d_min else None,
                                             "frac_of_h2d_ceiling": ((C_bytes / 1e9) / (-neg_h2d_min) * 1e3) / e2e_ms_max if neg_h2d_min else None,
                                             "numa": numa},
            "gpu_launches": int((stats["inflate_launches"] + stats["other_launches"]) * args.steps),
            "clocks": clocks, "parity": parity, "sample_parity": sample_parity, "merged_parity": merged_parity,
        }
        emit(line)
    lib.ngsq_host_free(pin_ptr)
    if N > 1:
        dist.destroy_process_group()
    for v in (parity_failed, merged_parity, sample_parity):
        if v and v.startswith("FAILED"):
            raise SystemExit("parity check failed: " + v)


if __name__ == "__main__":
    main()
