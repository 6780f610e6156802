"""BAM files with several read groups on several GPUs: `bamqualcheck --devices` on a 4-lane file and on a single-lane file
of the same size (cfg-3-like: 2x150bp, long-insert library on chr1-2 of GRCh38), cut into 1, 2, 4 and 8 pieces, one
per GPU (with fewer GPUs the pieces share them, up to 4 pieces), and the device time of the per-lane coverage shard
resolution (bqc_profile_read family 3: the lane split plus every lane's function and run) of the 4-lane file cut into
the same pieces in one process.  Checks that the .bamqc is the same for every piece count and prints one JSON line.
    python profiles/probes/lanes_devices_probe.py [records] [out_dir]"""
import json
import os
import re
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch

import bench
from bamqc_b200 import Engine, dist, synth

records_total = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
out_dir = sys.argv[2] if len(sys.argv) > 2 else None
n_gpus = torch.cuda.device_count()
props = torch.cuda.get_device_properties(0)
power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.split("\n")[0].strip()
# pieces per run: one per GPU; with fewer GPUs than pieces the pieces share the GPUs (a test of the cut, not of scaling)
counts = [n for n in (1, 2, 4, 8) if n <= max(n_gpus, 4)]
exe = os.path.join(ROOT, "bamqc_b200", "bin", "bamqualcheck")
result = dict(probe="lanes_devices", gpu=props.name, power_limit=power, n_gpus=n_gpus, records=None, files={})

with tempfile.TemporaryDirectory() as td:
    for n_lanes in (4, 1):
        spec = bench.workload_spec("cfg3", 1, records_total)
        spec["lib"] = dict(spec["lib"], n_lanes=n_lanes)
        spec["names"], spec["lengths"] = spec["names"][:2], spec["lengths"][:2]   # the reads lie on chr1-2 only
        genome, records, offsets = bench.make_workload(spec, 0, 1, records_total)
        header = synth.Library(n_lanes=n_lanes)
        fasta, bam = os.path.join(td, "g.fa"), os.path.join(td, f"lanes{n_lanes}.bam")
        if not os.path.exists(fasta):
            genome.write_fasta(fasta)
        synth.write_bam(bam, genome, header, records, int(offsets[-1]), level=1)
        n_rec = len(offsets) - 1
        result["records"] = n_rec
        row = dict(n_lanes=n_lanes, records=n_rec, file_mb=round(os.path.getsize(bam) / 2 ** 20, 1), runs={})
        outs = {}
        for n in counts:
            out = os.path.join(td, f"lanes{n_lanes}_n{n}.bamqc")
            best = None
            for rep in range(2):   # the first run of a device count also pays for reading the file from disk
                g = subprocess.run([exe, "-r", fasta, "-c", "chr1,chr2", "-i", "3000", "-o", out, "--timing", "--devices", ",".join(str(i % n_gpus) for i in range(n)), bam],
                                   capture_output=True, text=True)
                assert g.returncode == 0, g.stderr
                m = re.search(r"BAMQC_TIMING .*total_s=([0-9.]+) .*devices=(\d+)", g.stderr)
                assert m and int(m.group(2)) == n, g.stderr
                best = min(best or 1e9, float(m.group(1)))
            outs[n] = open(out).read()
            row["runs"][str(n)] = dict(gpus=min(n, n_gpus), total_s=best, m_records_per_s=round(n_rec / best / 1e6, 1))
        assert all(outs[n] == outs[counts[0]] for n in counts), "the .bamqc differs between device counts"
        if out_dir:
            os.makedirs(out_dir, exist_ok=True)
            open(os.path.join(out_dir, f"lanes{n_lanes}.bamqc"), "w").write(outs[counts[0]])
        if n_lanes > 1:
            # the same file cut into as many pieces as the last run in one process (pieces on the GPUs in turn): device time of the
            # per-lane shard resolution
            k = counts[-1]
            bounds = [n_rec * i // k for i in range(k + 1)]
            engines = []
            for i in range(k):
                e = Engine(lane_ids=synth.lane_ids(header), ref_names=genome.names, chroms="chr1,chr2", isize=3000, device=i % n_gpus)
                for rid, (p, m) in enumerate(zip(genome.packed, genome.lengths)):
                    e.set_reference(rid, p, m)
                e.cov_defer(2 if i == 0 else 1)
                for a in range(bounds[i], bounds[i + 1], 1 << 19):
                    o = offsets[a:min(bounds[i + 1], a + (1 << 19)) + 1]
                    e.submit(records[int(o[0]):int(o[-1])], o - o[0])
                e.finish()
                e.profile_enable(True)
                e.profile_read()
                engines.append(e)
            t0 = time.time()
            dist.resolve_coverage_local_lanes(engines, n_lanes)
            wall = time.time() - t0
            fam3 = [e.profile_read()["k_cov"][0] for e in engines]
            row["shard_resolution"] = dict(pieces=k, device_ms_per_piece=[round(x, 3) for x in fam3], wall_s=round(wall, 4),
                                           collected_records=[sum(int(e.cov_shard_boundary(lane).n) for lane in range(n_lanes)) for e in engines[1:]])
            for e in engines:
                e.close()
        result["files"]["lanes%d" % n_lanes] = row
        records = offsets = None
print(json.dumps(result))
