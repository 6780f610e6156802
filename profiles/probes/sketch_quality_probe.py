"""k_sketch time (CUDA events per launch group, serialised) per 10 M records on the standard library at -q 2, 3, 17 and
30 and on the stress() low-quality library at -q 17.  The share of valid 32-base windows, and with it the sub-chunks
k_sketch32v2 has to hash, goes from 100 % (-q 2) to ~50 % (-q 3), ~9 % (-q 17), ~0.1 % (-q 30) and 0 (stress).
python profiles/probes/sketch_quality_probe.py [n_pairs] [out.jsonl]"""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import torch
from bamqc_b200 import Engine, synth
n_pairs = int(sys.argv[1]) if len(sys.argv) > 1 else 1_000_000
out = sys.argv[2] if len(sys.argv) > 2 else ""
genome = synth.Genome.make(5, ["chr1", "chr2"], [40_000_000, 20_000_000])
for name, lib_, qs in (("standard", synth.Library(seed=9, n_pairs=n_pairs), (2, 3, 17, 30)),
                       ("stress", synth.Library(seed=9, n_pairs=n_pairs).stress(), (17,))):
    records, offsets = synth.generate(genome, lib_)
    n_rec = len(offsets) - 1
    for q in qs:
        eng = Engine(lane_ids=synth.lane_ids(lib_), ref_names=genome.names, chroms="chr1,chr2", qlist=(q,))
        for rid, (p, n) in enumerate(zip(genome.packed, genome.lengths)):
            eng.set_reference(rid, p, n)
        b = eng.prepare(records[:int(offsets[-1])], offsets)
        eng.profile_enable(2)
        ms = []
        for it in range(7):
            eng.reset(); eng.profile_read(); eng.run(b); eng.finish(); torch.cuda.synchronize()
            ms.append(eng.profile_read()["k_sketch"][0])
        ms = sorted(ms[2:])
        res = {"library": name, "q": q, "records": n_rec, "gpu": torch.cuda.get_device_name(0),
               "k_sketch_ms_per_10M_median": round(ms[len(ms) // 2] * 1e7 / n_rec, 3), "k_sketch_ms_per_10M_min": round(ms[0] * 1e7 / n_rec, 3)}
        print(json.dumps(res), flush=True)
        if out:
            with open(out, "a") as f:
                f.write(json.dumps(res) + "\n")
        eng.close()
