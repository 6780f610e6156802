"""SAM text on stdin (`bamqualcheck … -`, DESIGN §4.3): a cfg-2-like SAM file (2x150bp, GRCh38 contig lengths) written
by the C generator (bqc_synth_write_sam), read by the command through a pipe (`cat f.sam |`) and through redirected
stdin, and the same records as a BGZF BAM file for context (best of two runs each, BAMQC_TIMING).  Also the device time
of the SAM kernels per GB of text (bqc_profile_read family 10, in-process Engine.submit_sam in 256 MB submissions cut at
line ends) and the host encoder's rate on the same file on one thread of this box (tests/sam_selftest.cpp --time:
sam_line_to_bam, the encoder the command used before).  Checks that the three .bamqc files are identical and that no
line fell back to the host encoder.  Prints one JSON line.
    python profiles/probes/sam_probe.py [records] [out_dir]"""
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import torch

import bench
from bamqc_b200 import Engine, synth

records_total = int(sys.argv[1]) if len(sys.argv) > 1 else 10_000_000
out_dir = sys.argv[2] if len(sys.argv) > 2 else None
props = torch.cuda.get_device_properties(0)
power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.split("\n")[0].strip()
exe = os.path.join(ROOT, "bamqc_b200", "bin", "bamqualcheck")
result = dict(probe="sam", gpu=props.name, power_limit=power, host_cpu=os.cpu_count())


def timing(stderr):
    m = re.search(r"BAMQC_TIMING records=(\d+) .*total_s=([0-9.]+).*", stderr)
    assert m, stderr
    host = re.search(r"sam_host_lines=(\d+)", stderr)
    return int(m.group(1)), float(m.group(2)), int(host.group(1)) if host else None


with tempfile.TemporaryDirectory() as td:
    spec = bench.workload_spec("cfg2", 1, records_total)
    genome, records, offsets = bench.make_workload(spec, 0, 1, records_total)
    header = synth.Library()
    fasta, sam, bam = os.path.join(td, "g.fa"), os.path.join(td, "in.sam"), os.path.join(td, "in.bam")
    genome.write_fasta(fasta)
    synth.write_sam(sam, genome, header, records, int(offsets[-1]))
    synth.write_bam(bam, genome, header, records, int(offsets[-1]), level=1)
    n_rec = len(offsets) - 1
    sam_bytes = os.path.getsize(sam)
    result.update(records=n_rec, sam_gb=round(sam_bytes / 1e9, 3), bam_gb=round(os.path.getsize(bam) / 1e9, 3))
    records = offsets = None
    runs = {"sam_pipe": f"cat {sam} | {exe} -r {fasta} -o {td}/pipe.bamqc --timing -",
            "sam_redirect": f"{exe} -r {fasta} -o {td}/redirect.bamqc --timing - < {sam}",
            "bgzf_bam": f"{exe} -r {fasta} -o {td}/bam.bamqc --timing {bam}"}
    for name, cmd in runs.items():
        best = None
        for rep in range(2):
            g = subprocess.run(["bash", "-c", cmd], capture_output=True, text=True)
            assert g.returncode == 0, g.stderr
            n, total, host = timing(g.stderr)
            assert n == n_rec, g.stderr
            assert host in (None, 0), g.stderr
            best = min(best or 1e9, total)
        result[name] = dict(total_s=best, m_records_per_s=round(n_rec / best / 1e6, 2), text_gb_per_s=round(sam_bytes / best / 1e9, 3) if name != "bgzf_bam" else None)
    outs = [open(os.path.join(td, f)).read() for f in ("pipe.bamqc", "redirect.bamqc", "bam.bamqc")]
    assert outs[0] == outs[1] == outs[2], "the .bamqc differs between SAM and BAM input"
    if out_dir:
        os.makedirs(out_dir, exist_ok=True)
        open(os.path.join(out_dir, "sam_probe.bamqc"), "w").write(outs[0])

    # device time of the SAM kernels per GB of text, in process
    text = open(sam, "rb").read()
    body_at = 0
    while text[body_at:body_at + 1] == b"@":
        body_at = text.index(b"\n", body_at) + 1
    eng = Engine(lane_ids=synth.lane_ids(header), ref_names=genome.names)
    for rid, (p, m) in enumerate(zip(genome.packed, genome.lengths)):
        eng.set_reference(rid, p, m)
    eng.profile_enable(True)
    chunk = 256 << 20
    a, n_sub = body_at, 0
    while a < len(text):
        c = text.rfind(b"\n", a, a + chunk) + 1 if a + chunk < len(text) else len(text)
        eng.submit_sam(memoryview(text)[a:c], last=c == len(text))
        a, n_sub = c, n_sub + 1
    eng.finish()
    prof = eng.profile_read()
    assert eng.sam_host_lines == 0 and eng.records_seen == n_rec
    eng.close()
    text_gb = (len(text) - body_at) / 1e9
    result["k_sam"] = dict(submissions=n_sub, device_ms=round(prof["k_sam"][0], 2), ms_per_gb=round(prof["k_sam"][0] / text_gb, 2),
                           gb_per_s=round(text_gb / (prof["k_sam"][0] / 1e3), 1))
    text = None

    # the host encoder on the same file, one thread
    st = os.path.join(td, "sam_selftest")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", st, os.path.join(ROOT, "tests", "sam_selftest.cpp")], check=True)
    h = subprocess.run([st, "--time", sam], capture_output=True, text=True)
    assert h.returncode == 0, h.stdout + h.stderr
    host = json.loads(h.stdout)
    result["host_encoder_1_thread"] = dict(seconds=host["seconds"], m_lines_per_s=round(host["mlines_per_s"], 3), text_mb_per_s=round(host["mb_per_s"], 1))
    result["sam_pipe_vs_host_encoder"] = round(result["sam_pipe"]["m_records_per_s"] / host["mlines_per_s"], 1)
print(json.dumps(result))
