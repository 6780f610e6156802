#!/usr/bin/env python
"""bench.py -- BAM records/s of the per-record statistics pass (BASELINE.json metric) on N B200s.

A "step" is one whole pass of the hot path over the synthetic workload: reset, every record batch through
k_stats / k_eightmer / k_sketch and the coverage kernels (anchor recurrence included: nothing of the path runs on
the host), end-of-run flush and, for N > 1, the coverage shard protocol + the NCCL merge.
`value` is kernel-side throughput with the inflated record batches already in HBM; `e2e` is the same job through
the C ABI from pinned HOST buffers (H2D, device-side record framing, kernels, D2H of the result block).

Workloads (BASELINE.json configs, SURVEY 8d):
  cfg1  1 M records on a 10 Mb chr1                      (correctness size; also the GPU-vs-reference parity gate)
  cfg2  10 M records over chr1..22,X,Y, 1 GPU            (default at N = 1: the configuration the metric is quoted on)
  cfg3  100 M records on chr1-2, -i 3000, ONE stream cut into N contiguous pieces (default at N > 1; strong scaling)
  cfg4  high-error / low-quality library on the cfg1 geometry
  cfg5  --sweep: kernel-only on pre-inflated batches of 64 MB .. 8 GB

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config auto|cfg1|cfg2|cfg3|cfg4] [--records R]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "bam_records_per_second"
UNIT = "records/s"
HBM_FALLBACK_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback
DEFAULT_CHROMS = ",".join("chr%d" % i for i in range(1, 23))


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# Libraries (NCCL, torchrun) write banners to file descriptor 1; the contract is ONE JSON line on stdout.
# Everything written to fd 1 while the benchmark runs is redirected to stderr, the line goes to the real stdout.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit(line):
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return HBM_FALLBACK_GBS, "fallback"


# ------------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------------
def workload_spec(name, n_gpus, records=None):
    """Everything that defines a workload; identical for the b200 and the reference arm (`config` of the JSON line)."""
    from bamqc_b200 import synth
    if name == "auto":
        name = "cfg2" if n_gpus == 1 else "cfg3"
    if name in ("cfg1", "cfg4"):
        spec = dict(name=name, seed=20260101 if name == "cfg1" else 20260104, names=["chr1"], lengths=[10_000_000], active=[0],
                    records=1_000_000, isize=1000, lib={}, stress=name == "cfg4", scaling="strong",
                    what="synthetic 2x150bp records on a 10 Mb chr1" + (", high-error / low-quality library (5% mismatch, 30% soft-clipped, "
                                                                          "15% indel reads, MAPQ uniform)" if name == "cfg4" else ""))
    elif name == "cfg2":
        spec = dict(name=name, seed=20260102, names=list(synth.GRCH38_NAMES), lengths=list(synth.GRCH38), active=list(range(24)),
                    records=10_000_000, isize=1000, lib={}, stress=False, scaling="weak",
                    what="synthetic 2x150bp records over chr1..22,X,Y with GRCh38 lengths (3.09 Gb 2-bit reference in HBM per GPU)")
    elif name == "cfg3":
        spec = dict(name=name, seed=20260103, names=list(synth.GRCH38_NAMES), lengths=list(synth.GRCH38), active=[0, 1],
                    records=100_000_000, isize=3000, lib=dict(ins_mean=1500.0, ins_sd=400.0, ins_min=150, ins_max=6000), stress=False,
                    scaling="strong", what="synthetic 2x150bp records confined to chr1,chr2 (~30x), long-insert library, one stream cut into "
                                           "contiguous pieces, one per GPU")
    else:
        raise SystemExit("unknown --config " + name)
    if records:
        spec["records"] = int(records)
    # cfg2 keeps the historical meaning of --records: per GPU (weak scaling); the others are totals split N ways
    spec["records_per_gpu"] = spec["records"] if spec["scaling"] == "weak" else spec["records"] // n_gpus
    spec["records_total"] = spec["records_per_gpu"] * n_gpus
    spec["options"] = f"-k 32 -q 17 -e 0.01 -s 1 -i {spec['isize']} -c chr1..chr22"
    return spec


def config_of(spec, n_gpus):
    return {"workload": f"{spec['name']}: {spec['records_total']} {spec['what']}", "config": spec["name"], "records_total": spec["records_total"],
            "n_gpus": n_gpus, "options": spec["options"]}


def piece_regions(spec, piece, n_pieces):
    """Contiguous slice `piece` of the active genome (contigs in order, cut by cumulative length): {contig: (begin, end)}."""
    total = sum(spec["lengths"][c] for c in spec["active"])
    lo, hi = total * piece // n_pieces, total * (piece + 1) // n_pieces
    out, base = {}, 0
    for c in spec["active"]:
        n = spec["lengths"][c]
        a, b = max(lo, base), min(hi, base + n)
        if b > a:
            out[c] = (a - base, b - base)
        base += n
    return out


def available_host_gb():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable"):
                return int(line.split()[1]) / 1e6
    except Exception:
        pass
    return 1e9


def make_workload(spec, piece, n_pieces, n_records, threads=8, seed_shift=0):
    """Records of slice `piece`: generated in parallel sub-slices (ctypes releases the GIL).  Inside a slice the
    sub-slices are separated by ins_max + 1000 bp without fragment starts so that the slice is coordinate sorted; there
    is NO such hole between the slices of different pieces (the pieces are cut out of one stream)."""
    from bamqc_b200 import synth
    lengths = spec["lengths"]
    t0 = time.time()
    genome = synth.Genome.make(spec["seed"], spec["names"], lengths)
    regions = piece_regions(spec, piece, n_pieces)
    lib_kw = dict(spec["lib"])
    hole = int(lib_kw.get("ins_max", 1000)) + 1000
    total = sum(hi - lo for lo, hi in regions.values())
    n_pairs = int(n_records / 2.01)
    pieces = []
    target = max(total // (threads * 3), 1)
    for c in sorted(regions):
        lo, hi = regions[c]
        k = max(1, (hi - lo) // target)
        for j in range(k):
            a = lo + (hi - lo) * j // k
            b = lo + (hi - lo) * (j + 1) // k
            if j > 0:
                a += hole
            if b - a > 2 * hole:
                pieces.append((c, a, b))
    span = sum(b - a for _, a, b in pieces)
    results = [None] * len(pieces)
    pair_base = piece * 10 ** 8

    def work(i):
        c, a, b = pieces[i]
        lib_ = synth.Library(seed=spec["seed"] * 1000 + piece * 100000 + i + seed_shift, n_pairs=max(1, int(n_pairs * (b - a) / span)),
                             first_pair_id=pair_base + int(n_pairs * 1.05 * sum(q[2] - q[1] for q in pieces[:i]) / span),
                             regions={c: (a, b)}, **lib_kw)
        if spec["stress"]:
            lib_.stress()
        results[i] = synth.generate(genome, lib_)

    idx = list(range(len(pieces)))
    ths = [threading.Thread(target=lambda ids=idx[t::threads]: [work(i) for i in ids]) for t in range(threads)]
    [t.start() for t in ths]
    [t.join() for t in ths]
    # concatenate; both-unmapped tails (rID == -1) of every sub-slice move to the end as in a real BAM
    body, tails = [], []
    for rec, offs in results:
        n = len(offs) - 1
        k = n
        while k > 0 and rec[int(offs[k - 1]) + 4: int(offs[k - 1]) + 8].view(np.int32)[0] == -1:
            k -= 1
        body.append((rec, offs, 0, k))
        if k < n:
            tails.append((rec, offs, k, n))
    parts = body + tails
    n_rec = sum(e - s for _, _, s, e in parts)
    n_bytes = sum(int(o[e]) - int(o[s]) for _, o, s, e in parts)
    records = np.zeros(n_bytes + 64, dtype=np.uint8)
    offsets = np.zeros(n_rec + 1, dtype=np.uint64)
    p = r = 0
    for i, (rec, o, s, e) in enumerate(parts):
        nb = int(o[e]) - int(o[s])
        records[p:p + nb] = rec[int(o[s]):int(o[e])]
        offsets[r:r + (e - s)] = o[s:e] - o[s] + np.uint64(p)
        p += nb
        r += e - s
        parts[i] = None
    results = None
    offsets[n_rec] = p
    log(f"[piece {piece}/{n_pieces}] workload {spec['name']}: {n_rec} records, {n_bytes / 1e9:.3f} GB inflated, genome {sum(lengths) / 1e9:.2f} Gb, "
        f"{len(pieces)} sub-slices, {time.time() - t0:.1f}s")
    return genome, records, offsets


def split_batches(offsets, max_bytes):
    """Record index boundaries of batches of at most max_bytes."""
    bounds = [0]
    n = len(offsets) - 1
    while bounds[-1] < n:
        lo = bounds[-1]
        hi = int(np.searchsorted(offsets, offsets[lo] + np.uint64(max_bytes), side="right")) - 1
        bounds.append(max(lo + 1, min(hi, n)))
    return bounds


class ClockSampler:
    """SM clock and throttle reasons sampled while the bench runs (NVML from a thread every ~4 ms; `nvidia-smi -lms`
    cannot go below tens of milliseconds and missed the ~100 ms timed region).  mark() is called when the timed
    region starts: stop() reports the samples taken from then on (all samples if there were none)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        self.samples = []          # (time, sm_mhz, reasons bitmask)
        self.max_mhz = None
        self.t_mark = None
        self._halt = threading.Event()
        self.thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            try:
                import torch
                uuid = str(torch.cuda.get_device_properties(index).uuid)
                h = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            def loop():
                while not self._halt.is_set():
                    try:
                        self.samples.append((time.perf_counter(), float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)),
                                             int(pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h))))
                    except Exception:
                        pass
                    self._halt.wait(0.004)
            self.thread = threading.Thread(target=loop, daemon=True)
            self.thread.start()
        except Exception:
            self.thread = None

    def mark(self):
        self.t_mark = time.perf_counter()

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": []}
        if not self.thread:
            return out
        self._halt.set()
        self.thread.join(timeout=2)
        timed = [x for x in self.samples if self.t_mark is not None and x[0] >= self.t_mark]
        use = timed or self.samples
        if use:
            mask = 0
            for x in use:
                mask |= x[2]
            out = {"sm_mhz": statistics.median(x[1] for x in use), "sm_max_mhz": self.max_mhz,
                   "reasons": sorted(n for b, n in self.REASONS.items() if mask & b), "samples": len(use),
                   "sampled": "timed region" if timed else "warm-up + timed region", "how": "NVML, 4 ms period"}
        return out


# ------------------------------------------------------------------------------------------------------
# CPU side: the reference's own statistics code (oracle/_ref) or the oracle port, on host cores
# ------------------------------------------------------------------------------------------------------
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "bamqualcheck_ref")
CLI_BIN = os.path.join(ROOT, "bamqc_b200", "bin", "bamqualcheck")


def write_sample(genome, spec, records, offsets, lo, hi, td, tag):
    """Records [lo, hi) of the workload as a raw BAM + a FASTA with the contigs they lie on (in BAM order: the
    reference's FASTA cursor only moves forward, src/TripletCounting.hpp:255-259)."""
    from bamqc_b200 import synth

    def rid(i):
        return int(records[int(offsets[i]) + 4: int(offsets[i]) + 8].view(np.int32)[0])
    rids = sorted({rid(i) for i in (lo, hi - 1)} | {rid(i) for i in range(lo, hi, max(1, (hi - lo) // 64))})
    first = min([r for r in rids if r >= 0], default=0)
    last = max([r for r in rids if r >= 0], default=first)
    keep = list(range(first, last + 1))
    sub = synth.Genome([genome.names[c] for c in keep], [genome.lengths[c] for c in keep], [genome.packed[c] for c in keep])
    fasta = os.path.join(td, f"{tag}.fa")
    bam = os.path.join(td, f"{tag}.ubam")
    sub.write_fasta(fasta)
    a, b = int(offsets[lo]), int(offsets[hi])
    synth.write_bam(bam, genome, synth.Library(), records[a:b], b - a)
    return bam, fasta, hi - lo


def run_oracle_timed(bam, fasta, out, isize):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import bqc_testutil as util
    r = subprocess.run([util.ensure_oracle(), "-r", fasta, "-i", str(isize), "-o", out, "--timing", bam], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("oracle failed: " + r.stderr[-500:])
    for line in r.stderr.split("\n"):
        if line.startswith("ORACLE_TIMING"):
            kv = dict(x.split("=") for x in line.split()[1:])
            return int(kv["records"]), float(kv["loop_seconds"])
    raise RuntimeError("no timing line from the oracle")


def run_cpu_timed(bam, fasta, out, n_records, isize):
    """(records, seconds, kind).  kind "reference": oracle/_ref/bamqualcheck_ref = the reference's own
    src/bamqualcheck.cpp + statistics headers compiled unmodified over the SeqAn stand-in (whole process wall
    clock: raw BAM read, lazy FASTA load, statistics loop, output).  kind "port": the oracle restatement
    (statistics loop only) when the reference build is not in the tree."""
    if os.path.exists(REF_BIN):
        t0 = time.perf_counter()
        r = subprocess.run([REF_BIN, "-r", fasta, "-i", str(isize), "-o", out, bam], capture_output=True, text=True)
        dt = time.perf_counter() - t0
        if r.returncode == 0:
            return n_records, dt, "reference"
        log("reference build failed, falling back to the oracle port: " + r.stderr[-300:])
    n, s = run_oracle_timed(bam, fasta, out, isize)
    return n, s, "port"


def first_contig_prefix(records, offsets, max_records):
    """Record count of the longest prefix of at most max_records records that stays on the first contig."""
    n = min(max_records, len(offsets) - 1)

    def rid(i):
        return int(records[int(offsets[i]) + 4: int(offsets[i]) + 8].view(np.int32)[0])
    first_c = rid(0)
    if rid(n - 1) != first_c:
        lo, hi = 0, n - 1
        while hi - lo > 1:
            mid = (lo + hi) // 2
            if rid(mid) == first_c:
                lo = mid
            else:
                hi = mid
        n = hi
    return n


# ------------------------------------------------------------------------------------------------------
def dist_setup(world):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29511")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", local))
    return rank, local


def make_engine(spec, genome, local, staging_mb):
    from bamqc_b200 import Engine
    eng = Engine(lane_ids=["L1"], ref_names=genome.names, isize=spec["isize"], klist=(32,), qlist=(17,), e=0.01, seed=1,
                 device=local, staging_bytes=staging_mb << 20)
    for rid, (p, n) in enumerate(zip(genome.packed, genome.lengths)):
        eng.set_reference(rid, p, n)
    return eng


def all_tables(eng, dev):
    """The whole result block (every counter of every table) + the sketch as device tensors, for exact comparisons."""
    import torch
    c = torch.empty(eng.counters_len(), dtype=torch.int64, device=dev)
    s = torch.empty(max(1, eng.sketch_len()), dtype=torch.uint8, device=dev)
    eng.export_to(c.data_ptr(), s.data_ptr())
    torch.cuda.synchronize(dev)
    return c, s


DUMP_LIMIT_BYTES = 64 << 20


def result_arrays(eng):
    """What a caller of the engine receives after bqc_finish, as float64 arrays that hold every value exactly: each
    result table of each lane (per mate for the per-cycle fields, per q/k pair for the k-mer fields), the per-cycle mean
    qualities, the KmerStream estimators, and the packed sketch words split into their low and high 32 bits (the words
    are bit sets and do not fit a double's 53-bit mantissa)."""
    from bamqc_b200.engine import FIELDS
    n_qk = len(eng.klist) * len(eng.qlist)
    out = {}
    for lane in range(len(eng.lane_ids)):
        for name, f in FIELDS.items():
            if f >= FIELDS["SUMCOUNT"]:
                subs = [(f"_qk{i}", i) for i in range(n_qk)]
            elif f >= FIELDS["READLEN"]:
                subs = [("_mate0", 0), ("_mate1", 1)]
            else:
                subs = [("", 0)]
            for suffix, sub in subs:
                t = eng.table(name, lane, sub)
                if t.size and int(t.max()) >= 1 << 53:
                    raise RuntimeError(f"lane {lane} {name}{suffix}: a count of 2**53 or more has no exact float64")
                out[f"lane{lane}_{name}{suffix}"] = t.astype(np.float64)
        for mate in (0, 1):
            out[f"lane{lane}_avgqual_mean_mate{mate}"] = eng.avgqual(lane, mate).astype(np.float64)
        for qk in range(n_qk):
            est = eng.estimates(lane, qk)
            out[f"lane{lane}_estimates_qk{qk}"] = np.array([est[k] for k in ("sumCount", "F0", "f1", "F2")], dtype=np.float64)
            words = eng.sketch(lane, qk)
            out[f"lane{lane}_sketch_qk{qk}"] = np.stack([words & np.uint64(0xFFFFFFFF), words >> np.uint64(32)], axis=1).astype(np.float64)
    return out


def dump_outputs(eng, out_dir):
    """--dump-outputs: one <name>.npy per result array (result_arrays), at most DUMP_LIMIT_BYTES in all."""
    arrays = result_arrays(eng)
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes of results, more than the {DUMP_LIMIT_BYTES} allowed")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    log(f"dumped {len(arrays)} result arrays ({total / 1e6:.1f} MB) to {out_dir}")


def run_sweep(args):
    """cfg 5 of BASELINE.json: kernel-only throughput on pre-inflated record batches of 64 MB .. 8 GB resident in HBM
    (one GPU, or one slice per rank under torchrun).  One JSON line per size: median and best of --steps repetitions,
    CUDA events on the engine's stream.  Sizes below the L2 capacity are flagged (their inputs can sit in L2)."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = dist_setup(world)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    spec = workload_spec("cfg2", world)
    sizes_mb = [int(x) for x in args.sweep.split(",")]
    top = max(sizes_mb) << 20
    genome, records, offsets = make_workload(spec, rank, world, int(top / 290.0) + 1000, threads=args.threads)
    eng = make_engine(spec, genome, local, args.staging_mb)
    stream = torch.cuda.ExternalStream(eng.stream, device=dev)
    for mb in sizes_mb:
        want = mb << 20
        k = int(np.searchsorted(offsets, want, side="right")) - 1
        k = max(1, min(k, len(offsets) - 1))
        sub = offsets[:k + 1]
        bounds = split_batches(sub, args.batch_mb << 20)
        batches = []
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            o = sub[lo:hi + 1]
            batches.append(eng.prepare(records[int(o[0]):int(o[-1])], o - o[0]))
        times = []
        reps = args.steps
        for it in range(args.warmup + reps):
            torch.cuda.synchronize(dev)
            if world > 1:
                dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            eng.reset()
            for b in batches:
                eng.run(b)
            eng.finish()
            e1.record(stream)
            torch.cuda.synchronize(dev)
            if it >= args.warmup:
                times.append(e0.elapsed_time(e1))
        for b in batches:
            b.free()
        t = torch.tensor([float(np.median(times)), float(min(times))], dtype=torch.float64, device=dev)
        tot = torch.tensor([float(k), float(sub[-1])], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        med, best = float(t[0].item()), float(t[1].item())
        if rank == 0:
            emit({"sweep": "cfg5: kernel-only, pre-inflated resident batches (independent slices, no cross-GPU step)", "batch_mb_per_gpu": mb, "n_gpus": world,
                  "records": int(tot[0].item()), "bytes": int(tot[1].item()), "reps": reps, "ms_median": med, "ms_best": best,
                  "records_per_s_median": tot[0].item() / (med / 1e3), "records_per_s_best": tot[0].item() / (best / 1e3),
                  "gbs_median": tot[1].item() / (med / 1e3) / 1e9, "inputs_fit_l2": bool(sub[-1] < 120e6)})
    eng.close()
    if world > 1:
        dist.destroy_process_group()


def run_b200(args):
    import torch
    import torch.distributed as dist
    from bamqc_b200 import synth, dist as bdist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        log(f"warning: --gpus {args.gpus} but WORLD_SIZE {world}; using WORLD_SIZE")
    rank, local = dist_setup(world)
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    spec = workload_spec(args.config, world, args.records)
    # host memory: the piece, a transient copy while it is assembled, and the CPU sample; scale down rather than swap
    per_gpu = spec["records_per_gpu"]
    need_gb = per_gpu * 290 * 2.3 / 1e9 * min(world, 8)
    avail = available_host_gb()
    scaled = None
    if need_gb > 0.8 * avail:
        f = 0.8 * avail / need_gb
        scaled = f"records per GPU scaled by {f:.2f}: {need_gb:.0f} GB of host memory needed, {avail:.0f} GB available"
        if args.dump_outputs:  # dumps of two runs are comparable only if the arguments alone fix the inputs
            raise SystemExit(f"--dump-outputs: {need_gb:.0f} GB of host memory needed, {avail:.0f} GB available; "
                             "choose a smaller workload with --records instead of letting it be scaled down")
        log("warning: " + scaled)
        per_gpu = int(per_gpu * f)
        spec["records_per_gpu"], spec["records_total"] = per_gpu, per_gpu * world
    # one stream cut into `world` pieces when the workload is a single sample (cfg3); independent slices for cfg2 x N
    sharded = world > 1
    genome, records, offsets = make_workload(spec, rank, world, per_gpu, threads=args.threads)
    n_rec = len(offsets) - 1
    n_bytes = int(offsets[-1])

    eng = make_engine(spec, genome, local, args.staging_mb)
    log(f"[rank {rank}] reference in HBM: {sum(genome.lengths) / 4 / 1e6:.0f} MB 2-bit")
    exchange = bdist.torch_exchange(device=dev) if sharded else None

    def finish_step(bufs):
        """End of input on every rank: the pieces resolve the coverage windows across the cuts, then one all-reduce."""
        eng.finish()
        if sharded:
            delta = bdist.resolve_coverage_shards(eng, rank, exchange)
            bufs = bdist.reduce_engine(eng, bufs)
            eng.poscov_adjust(delta)
        return bufs

    # ---- resident batches (kernel-only) ---------------------------------------------------------------
    bounds = split_batches(offsets, args.batch_mb << 20)
    batches = []
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        o = offsets[lo:hi + 1]
        batches.append(eng.prepare(records[int(o[0]):int(o[-1])], o - o[0]))
    stream = torch.cuda.ExternalStream(eng.stream, device=dev)
    bufs = None

    def step():
        nonlocal bufs
        eng.reset()
        if sharded:
            eng.cov_defer(2 if rank == 0 else 1)
        for b in batches:
            eng.run(b)
        bufs = finish_step(bufs)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local) if rank == 0 else None  # sampled from the warm-up on (the timed region is short)
    for _ in range(args.warmup):
        step()
    eng.profile_enable(True)
    eng.profile_read()
    launches0 = eng.kernel_launches
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if sampler:
        sampler.mark()
    ev0.record(stream)
    for _ in range(args.steps):
        step()
    ev1.record(stream)
    barrier()
    ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if sampler else None
    launches = eng.kernel_launches - launches0
    prof = eng.profile_read()
    eng.profile_enable(False)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    tot = torch.tensor([float(n_rec), float(n_bytes)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms = float(t.item())
    total_records, total_bytes = float(tot[0].item()), float(tot[1].item())
    value = total_records * args.steps / (ms / 1e3)
    ref_tables = all_tables(eng, dev)
    if args.dump_outputs and rank == 0:  # every rank holds the merged result after the last timed step
        dump_outputs(eng, args.dump_outputs)

    # one more pass with the coverage kernels on the compute stream: exclusive device time per kernel family
    eng.profile_enable(2)
    eng.profile_read()
    step()
    serial = eng.profile_read()
    eng.profile_enable(False)
    fams = ("k_stats", "k_eightmer", "k_sketch", "k_cov")
    serial_ms = {f: serial[f][0] for f in fams}
    serial_sum = max(1e-9, sum(serial_ms.values()))

    # ---- end to end through the C ABI from pinned host buffers -----------------------------------------
    # the workload array itself is page-locked in place (no second copy of a multi-GB piece)
    cudart = torch.cuda.cudart()
    reg = cudart.cudaHostRegister(records.ctypes.data, records.nbytes, 0)
    pinned_how = "cudaHostRegister of the workload array" if int(reg) == 0 else "pageable (staged through the engine's pinned slots)"
    e2e_bounds = split_batches(offsets, (args.staging_mb << 20) - 4096)
    h2d = n_bytes
    d2h = eng.counters_len() * 8 + eng.sketch_len() // 2 + 48 * (len(e2e_bounds) - 1)

    def e2e_step():
        eng.reset()
        if sharded:
            eng.cov_defer(2 if rank == 0 else 1)
        for lo, hi in zip(e2e_bounds[:-1], e2e_bounds[1:]):
            o = offsets[lo:hi + 1]
            eng.submit(records[int(o[0]):int(o[-1])], None)  # the engine frames the records itself (on the device)
        finish_step(bufs)
        return eng.scalars()  # D2H of the result block

    e2e_steps = max(1, min(args.steps, 5))
    for _ in range(max(1, min(args.warmup, 4))):  # also cycles through all four staging slots (allocated on first use)
        e2e_step()
    barrier()
    eng.profile_enable(True)
    eng.profile_read()
    w0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = time.perf_counter() - w0
    e2e_prof = eng.profile_read()
    eng.profile_enable(False)
    log(f"[rank {rank}] e2e: {e2e_s / e2e_steps * 1e3:.1f} ms/step; device kernels "
        f"{sum(e2e_prof[k][0] for k in ('k_stats', 'k_eightmer', 'k_sketch')) / e2e_steps:.1f} ms, framing {e2e_prof['k_frame'][0] / e2e_steps:.1f} ms")
    te = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = total_records * e2e_steps / float(te.item())
    e2e_tables = all_tables(eng, dev)
    paths_agree = {"resident_vs_streaming": bool(torch.equal(ref_tables[0], e2e_tables[0]) and torch.equal(ref_tables[1], e2e_tables[1]))}

    # ---- end to end from BGZF-compressed host buffers (extra keys, not the contract's e2e) -------------------
    # e2e_bgzf: the compressed blocks go over PCIe and are inflated + framed on the device (bqc_submit_bgzf), every rank
    # its own piece; e2e_bgzf_host: zlib on the host threads (north_star's "host keeps BGZF inflate"), bounded sample
    bgzf = bgzf_host = None
    if args.bgzf_records != 0:
        k = n_rec if args.bgzf_records < 0 else min(args.bgzf_records, n_rec)
        raw = records[:int(offsets[k])]
        t0 = time.perf_counter()
        comp = synth.bgzf_compress(raw, level=args.bgzf_level)
        log(f"[rank {rank}] BGZF level {args.bgzf_level}: {raw.size / 1e6:.0f} MB -> {comp.size / 1e6:.0f} MB in {time.perf_counter() - t0:.1f}s")
        cpin = torch.empty(comp.size, dtype=torch.uint8, pin_memory=True)
        cpin.numpy()[:] = comp
        cnp = cpin.numpy()

        def bgzf_step():
            eng.reset()
            if sharded:
                eng.cov_defer(2 if rank == 0 else 1)
            eng.submit_bgzf(cnp, last=True)
            finish_step(bufs)
            return eng.scalars()

        for _ in range(2):
            bgzf_step()
        barrier()
        eng.profile_enable(True)
        eng.profile_read()
        reps = 3
        w0 = time.perf_counter()
        for _ in range(reps):
            bgzf_step()
        barrier()
        dt = (time.perf_counter() - w0) / reps
        bprof = eng.profile_read()
        eng.profile_enable(False)
        if k == n_rec:
            bt = all_tables(eng, dev)
            paths_agree["resident_vs_bgzf"] = bool(torch.equal(ref_tables[0], bt[0]) and torch.equal(ref_tables[1], bt[1]))
        inflate_ms = bprof["k_inflate"][0] / reps
        tb = torch.tensor([dt, float(k), float(comp.size)], dtype=torch.float64, device=dev)
        if world > 1:
            tmax = tb.clone()
            dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
            dist.all_reduce(tb, op=dist.ReduceOp.SUM)
            dt_all, k_all, comp_all = float(tmax[0].item()), float(tb[1].item()), float(tb[2].item())
        else:
            dt_all, k_all, comp_all = dt, float(k), float(comp.size)
        bgzf = {"value": k_all / dt_all, "unit": UNIT, "records": int(k_all), "ms_per_step": dt_all * 1e3, "compressed_mb": comp_all / 1e6, "level": args.bgzf_level,
                "h2d_bytes_per_step": int(comp_all), "k_inflate_ms_rank0": inflate_ms, "k_inflate_gbs_out_rank0": raw.size / max(1e-9, inflate_ms / 1e3) / 1e9,
                "k_frame_ms_rank0": bprof["k_frame"][0] / reps, "ranks": world,
                "path": "bqc_submit_bgzf on every rank: compressed blocks H2D, device inflate (warp per block), device framing, kernels, merge, D2H of results"}
        log(f"[rank {rank}] e2e_bgzf (device inflate): {dt * 1e3:.1f} ms for {k} records; k_inflate {inflate_ms:.1f} ms, framing {bgzf['k_frame_ms_rank0']:.1f} ms")
        if rank == 0 and world == 1:  # host zlib arm on a bounded sample
            kh = min(k, 800_000)
            rawh = records[:int(offsets[kh])]
            comph = comp if kh == k else synth.bgzf_compress(rawh, level=args.bgzf_level)
            stage_cap = args.staging_mb << 20
            if rawh.size <= stage_cap:
                eng.reset()
                w0 = time.perf_counter()
                out = eng.acquire_staging()
                n_inf = eng.lib.bqc_bgzf_inflate(comph.ctypes.data, comph.size, out.ctypes.data, min(out.size, stage_cap), args.threads)
                if n_inf:
                    eng.submit(out[:n_inf], None)
                    eng.finish()
                    eng.scalars()
                    dth = time.perf_counter() - w0
                    bgzf_host = {"value": kh / dth, "unit": UNIT, "records": kh, "threads": args.threads, "compressed_mb": comph.size / 1e6}
    if int(reg) == 0:
        cudart.cudaHostUnregister(records.ctypes.data)

    # ---- roofline of the dominant kernel (CUDA events on the launching stream, live) --------------------
    peak, which = measured_peak()
    fam = max(("k_stats", "k_eightmer", "k_sketch"), key=lambda f: prof[f][0])
    fam_ms, fam_n = prof[fam]
    per_launch_ms = fam_ms / max(1, fam_n)
    alg_bytes = n_bytes * args.steps / max(1, fam_n)  # algorithmic bytes one launch covers = inflated bytes of its batch
    achieved = alg_bytes / (per_launch_ms / 1e3) / 1e9 if per_launch_ms > 0 else 0.0
    traffic = traffic_src = None
    tfile = os.path.join(ROOT, "profiles", "r2", "traffic.json")
    if os.path.exists(tfile):
        try:
            tj = json.load(open(tfile))
            traffic, traffic_src = tj.get(fam), tj.get("_source")
        except Exception:
            traffic = None

    # ---- CPU baseline + parity gate (rank 0, N = 1 only) ------------------------------------------------
    # the reference's own statistics code on a bounded sample of the same workload, one thread; the product CLI then
    # reads the SAME two files on the GPU and the two .bamqc outputs must be byte-identical (every table, every double)
    cpu = parity = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        with tempfile.TemporaryDirectory() as td:
            k = first_contig_prefix(records, offsets, args.cpu_sample)
            bam, fasta, k = write_sample(genome, spec, records, offsets, 0, k, td, "cpu")
            ref_out = os.path.join(td, "cpu.bamqc")
            nrec_o, secs, kind = run_cpu_timed(bam, fasta, ref_out, k, spec["isize"])
            n_p, secs_p = run_oracle_timed(bam, fasta, os.path.join(td, "cpu_port.bamqc"), spec["isize"])
            what = ("oracle/_ref/bamqualcheck_ref (the reference's own sources over the SeqAn stand-in), whole process wall clock "
                    "on a raw BAM incl. FASTA load and output" if kind == "reference" else "oracle/bamqualcheck_oracle, statistics loop only")
            cpu = {"value": nrec_o / secs, "unit": UNIT, "cores": 1, "kind": kind,
                   "sample": f"first {nrec_o} records of the workload (one contig), single thread, {what}",
                   "port_loop_only": n_p / secs_p}
            gpu_out = os.path.join(td, "gpu.bamqc")
            t0 = time.perf_counter()
            r = subprocess.run([CLI_BIN, "-r", fasta, "-i", str(spec["isize"]), "-o", gpu_out, bam], capture_output=True, text=True)
            cli_s = time.perf_counter() - t0
            same = r.returncode == 0 and open(gpu_out, "rb").read() == open(ref_out, "rb").read()
            parity = {"identical": bool(same), "records": int(nrec_o), "lines": len(open(ref_out).read().split("\n")) - 1,
                      "gpu": "bamqc_b200/bin/bamqualcheck (the drop-in command) on the same BAM + FASTA", "against": what.split(",")[0],
                      "compared": "whole .bamqc byte for byte (every count table, estimator and per-cycle double)", "cli_seconds": cli_s}
            if not same:
                log("PARITY FAILURE: the GPU .bamqc differs from the reference's\n" + r.stderr[-500:])

    if rank == 0:
        cfg = config_of(spec, world)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": spec["scaling"], "vs_baseline": None,
            "dtype": "u8/u32/u64 integer", "data": "synthetic",
            "config": cfg,
            "engine": {"records_per_gpu": per_gpu, "inflated_gb_per_gpu": n_bytes / 1e9, "batches_per_gpu": len(batches), "batch_mb": args.batch_mb,
                       "l2": "inputs larger than L2 (no flush needed)" if n_bytes > 130e6 else "inputs may sit in L2",
                       "sharding": ("one stream cut into contiguous pieces (no re-anchoring gaps between pieces); coverage windows resolved across the "
                                    "cuts with the bqc_cov_shard_* protocol (3 small all-gathers), tables merged with one NCCL all-reduce") if sharded else "single GPU",
                       "timed_region": "reset, all batches through every kernel incl. the coverage anchor recurrence (device), end-of-run flush"
                                       + (", shard protocol, all-reduce" if sharded else ""),
                       "scaled_down": scaled},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                    "host_buffers": pinned_how,
                    "path": "bqc_submit from pinned host buffers: H2D, device-side record framing, all statistics kernels (nothing on the host), D2H of results"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": fam, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "peak_source": which, "traffic": traffic, "traffic_source": traffic_src, "alg_bytes_per_launch": alg_bytes, "ms_per_launch": per_launch_ms,
                         "serialised_ms_per_step": {f: round(v, 4) for f, v in serial_ms.items()},
                         "serialised_share": {f: round(v / serial_sum, 4) for f, v in serial_ms.items()},
                         "serialised_note": "one extra pass with the coverage kernels on the compute stream (bqc_profile_enable 2): exclusive CUDA-event "
                                            "time per kernel family, no overlap between families",
                         "all_kernels_gbs": n_bytes / (serial_sum / 1e3) / 1e9, "step_gbs": total_bytes / world / (ms / args.steps / 1e3) / 1e9},
            "cpu_baseline": cpu,
            "parity_checked": parity,
            "paths_agree": paths_agree,
        }
        if bgzf:
            line["e2e_bgzf"] = bgzf
        if bgzf_host:
            line["e2e_bgzf_host"] = bgzf_host
        emit(line)
    for b in batches:
        b.free()
    eng.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_reference(args):
    """Reference arm: the reference's own CPU implementation (oracle/_ref/bamqualcheck_ref, else the oracle port) on all
    host cores.  The program is single-threaded by construction, so the WHOLE workload is cut into `cores` contiguous
    record ranges and every step runs `cores` independent processes concurrently, each over its own range (>= 600 k
    records); a step lasts as long as its slowest process.  Imports only the synthetic generator (libbamqc_synth.so):
    no product code is loaded or run."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    cores = args.threads
    spec = workload_spec(args.config, world, args.records)
    cfg = config_of(spec, world)
    # bounded sample of the workload: at most --ref-records (default 10 M = all of cfg2) of piece 0
    total = min(spec["records_total"], args.ref_records)
    genome, records, offsets = make_workload(spec, 0, max(1, spec["records_total"] // total), total, threads=args.threads)
    n_rec = len(offsets) - 1
    with tempfile.TemporaryDirectory() as td:
        shards = []
        t0 = time.time()
        for c in range(cores):
            lo, hi = n_rec * c // cores, n_rec * (c + 1) // cores
            if hi > lo:
                shards.append(write_sample(genome, spec, records, offsets, lo, hi, td, f"s{c}"))
        log(f"reference arm: {len(shards)} processes x ~{n_rec // max(1, len(shards))} records, files written in {time.time() - t0:.1f}s")

        def one_step():
            res = [None] * len(shards)

            def w(i):
                res[i] = run_cpu_timed(shards[i][0], shards[i][1], os.path.join(td, f"o{i}.bamqc"), shards[i][2], spec["isize"])
            ths = [threading.Thread(target=w, args=(i,)) for i in range(len(shards))]
            t0 = time.perf_counter()
            [t.start() for t in ths]
            [t.join() for t in ths]
            return sum(r[0] for r in res), time.perf_counter() - t0, max(r[1] for r in res), res[0][2]

        for _ in range(args.warmup):
            one_step()
        tot_rec = tot_s = 0.0
        kind = "port"
        for _ in range(args.steps):
            n, wall, slowest, kind = one_step()
            tot_rec += n
            tot_s += slowest  # the processes run concurrently: a step lasts as long as its slowest process
        value = tot_rec / tot_s
        loop_only = None
        try:
            n_p, secs_p = run_oracle_timed(shards[0][0], shards[0][1], os.path.join(td, "port.bamqc"), spec["isize"])
            loop_only = n_p / secs_p
        except Exception:
            pass
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": tot_s / args.steps * 1e3, "higher_is_better": True, "scaling": spec["scaling"], "vs_baseline": None,
        "dtype": "u8/u32/u64 integer", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": len(shards), "kind": kind,
                         "sample": f"{int(tot_rec / args.steps)} records of the workload per step (a bounded sample when the workload is larger), cut into "
                                   f"{len(shards)} contiguous ranges, one single-threaded process each, all concurrent; " + (
                             "oracle/_ref/bamqualcheck_ref = the reference's own src/bamqualcheck.cpp + statistics headers compiled unmodified "
                             "over the SeqAn stand-in (SeqAn 1.4.2 is unavailable), whole process wall clock incl. FASTA load" if kind == "reference" else
                             "oracle/bamqualcheck_oracle (CPU restatement of the reference), statistics loop only"),
                         "one_thread_loop_only_port": loop_only},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="auto", choices=["auto", "cfg1", "cfg2", "cfg3", "cfg4"],
                    help="auto: cfg2 on one GPU (the configuration the metric is quoted on), cfg3 (100 M records cut across the GPUs) otherwise")
    ap.add_argument("--records", type=int, default=0, help="override the record count of the workload (cfg2: per GPU; others: total)")
    ap.add_argument("--batch-mb", type=int, default=1024)
    ap.add_argument("--staging-mb", type=int, default=256)
    ap.add_argument("--threads", type=int, default=min(16, os.cpu_count() or 8))
    ap.add_argument("--cpu-sample", type=int, default=1_500_000, help="records of the CPU baseline / parity sample")
    ap.add_argument("--ref-records", type=int, default=10_000_000, help="reference arm: records of the workload run per step")
    ap.add_argument("--bgzf-records", type=int, default=-1, help="records of the BGZF end-to-end measurement per GPU (0 = skip, < 0 = the whole piece)")
    ap.add_argument("--bgzf-level", type=int, default=6, help="zlib level of the synthetic BGZF input (samtools default: 6)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--sweep", default="", help="cfg 5: comma separated batch sizes in MB per GPU (e.g. 64,256,1024,4096,8192); prints one line per size")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write the results of the last one as DIR/<name>.npy (float64, exact)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.sweep):
        ap.error("--dump-outputs applies to the timed path of --impl b200 without --sweep")
    if args.warmup < 3 and args.impl == "b200":
        log("note: fewer than 3 warm-up steps requested; timing rules ask for >= 3")
    if args.impl == "reference":
        run_reference(args)
    elif args.sweep:
        run_sweep(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
