"""Shared helpers of the parity tests: build/run the CPU oracle (test infrastructure under oracle/),
make synthetic data sets, run the CUDA engine through the C ABI and diff the `.bamqc` outputs."""
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_BIN = os.path.join(ORACLE_DIR, "bamqualcheck_oracle")


def ensure_oracle():
    src = os.path.join(ORACLE_DIR, "bamqc_oracle.cpp")
    if not os.path.exists(ORACLE_BIN) or os.path.getmtime(ORACLE_BIN) < os.path.getmtime(src):
        subprocess.run(["make", "-C", ORACLE_DIR, "all"], check=True, capture_output=True)
    return ORACLE_BIN


def run_oracle(bam, fasta, out, chroms=None, isize=None, klist=None, qlist=None, e=None, seed=None, dump=None, extra=()):
    cmd = [ensure_oracle(), "-r", str(fasta), "-o", str(out)]
    if chroms is not None:
        cmd += ["-c", chroms]
    if isize is not None:
        cmd += ["-i", str(isize)]
    if klist is not None:
        cmd += ["-k", ",".join(map(str, klist))]
    if qlist is not None:
        cmd += ["-q", ",".join(map(str, qlist))]
    if e is not None:
        cmd += ["-e", repr(e)]
    if seed is not None:
        cmd += ["-s", str(seed)]
    if dump is not None:
        cmd += ["--dump", str(dump)]
    cmd += list(extra) + [str(bam)]
    return subprocess.run(cmd, capture_output=True, text=True)


def small_genome(seed=7, lengths=(400000, 300000, 100000), names=("chr1", "chr2", "chrX")):
    from bamqc_b200 import synth
    return synth.Genome.make(seed, list(names), list(lengths))


def diff_bamqc(a_path, b_path, max_report=8):
    """Return a list of human-readable differences between two .bamqc files (empty = identical)."""
    a = open(a_path).read().split("\n")
    b = open(b_path).read().split("\n")
    out = []
    if len(a) != len(b):
        out.append(f"line count {len(a)} vs {len(b)}")
    for i, (x, y) in enumerate(zip(a, b)):
        if x != y:
            xs, ys = x.split(" "), y.split(" ")
            key = xs[0]
            where = next((j for j, (p, q) in enumerate(zip(xs, ys)) if p != q), min(len(xs), len(ys)))
            out.append(f"line {i} key {key} len {len(xs)} vs {len(ys)} first diff at field {where}: "
                       f"{xs[where:where + 4]} vs {ys[where:where + 4]}")
            if len(out) >= max_report:
                break
    return out


def run_engine(genome, lib_, records, offsets, out_path, chroms="chr1,chr2", isize=1000, klist=(32,), qlist=(17,),
               e=0.01, seed=1, n_batches=1, sample_id="S1", resident=False, engine_kwargs=None, keep=False, mode="offsets",
               chunk_bytes=None):
    """Push `records` through the CUDA engine via the C ABI and write the .bamqc text.
    mode: "offsets" (host-framed, offsets given), "whole" (whole-record slices, framed by the engine),
    "stream" (arbitrary chunk_bytes-sized chunks of the byte stream through bqc_submit_stream)."""
    from bamqc_b200 import Engine, synth
    eng = Engine(lane_ids=synth.lane_ids(lib_), ref_names=genome.names, chroms=chroms, isize=isize, klist=klist,
                 qlist=qlist, e=e, seed=seed, **(engine_kwargs or {}))
    for rid, (p, n) in enumerate(zip(genome.packed, genome.lengths)):
        eng.set_reference(rid, p, n)
    nrec = len(offsets) - 1
    bounds = [nrec * i // n_batches for i in range(n_batches + 1)]
    batches = []
    if mode == "stream":
        total = int(offsets[-1])
        step = chunk_bytes or max(1, total // max(1, n_batches))
        p = 0
        while True:
            q = min(total, p + step)
            eng.submit_stream(records[p:q], last=q >= total)
            p = q
            if p >= total:
                break
        n_batches = 0
    for i in range(n_batches):
        lo, hi = bounds[i], bounds[i + 1]
        if hi == lo:
            continue
        o = offsets[lo:hi + 1]
        if resident:
            batches.append(eng.prepare(records[int(o[0]):int(o[-1])], o - o[0]))
        elif mode == "whole":
            eng.submit(records[int(o[0]):int(o[-1])], None)
        else:
            eng.submit(records, o)
    if resident:
        for rep in range(2):  # replay twice: results must come from the second, post-reset pass
            eng.reset()
            for b in batches:
                eng.run(b)
            eng.finish()
    else:
        eng.finish()
    eng.write_bamqc(sample_id, out_path)
    if keep:
        return eng
    for b in batches:
        b.free()
    eng.close()
    return None


def oracle_sketch_geometry(dump_path):
    """[(size, F2size, sumCount)] of every sketch in the oracle's dump, in dump order (lanes in std::map order, then
    q, then k): the `sketch_geometry` lines of oracle/bamqc_oracle.cpp (writeDump)."""
    out = []
    for line in open(dump_path):
        f = line.split()
        if f and f[0] == "sketch_geometry":
            out.append((int(f[3]), int(f[4]), int(f[5])))
    return out


def oracle_sketch(dump_path, n_sketches=None):
    """[(sketch table, F2 table)] of every sketch in the oracle's dump, sized by its `sketch_geometry` lines."""
    geo = oracle_sketch_geometry(dump_path)
    if n_sketches is not None:
        assert len(geo) == n_sketches
    raw = np.fromfile(str(dump_path) + ".sketch", dtype=np.uint64)
    assert raw.size == sum(32 * size + f2size for size, f2size, _ in geo)
    out, p = [], 0
    for size, f2size, _ in geo:
        out.append((raw[p:p + 32 * size], raw[p + 32 * size:p + 32 * size + f2size]))
        p += 32 * size + f2size
    return out


def assert_sketches_equal(eng, dump_path, lane_ids, n_qk):
    """Raw sketch, F2 table and sumCount of every (lane, q/k pair) of the engine equal to the oracle's dump."""
    sk = oracle_sketch(dump_path, len(lane_ids) * n_qk)
    geo = oracle_sketch_geometry(dump_path)
    i = 0
    for lane in sorted(range(len(lane_ids)), key=lambda l: lane_ids[l]):  # the oracle dumps lanes in std::map order
        for qk in range(n_qk):
            table, f2 = sk[i]
            assert np.array_equal(eng.sketch(lane, qk), table), f"sketch table lane {lane} qk {qk}"
            assert np.array_equal(eng.table("F2TABLE", lane, qk), f2), f"F2 table lane {lane} qk {qk}"
            assert eng.estimates(lane, qk)["sumCount"] == geo[i][2], f"sumCount lane {lane} qk {qk}"
            i += 1


def kernel_names(fn):
    """Run fn() under torch.profiler with CUDA activities; return (fn's result, the set of kernel names that ran).
    Demangled names look like `void bqc::k_sketch32v2<640u>(bqc::EngineView, ...)`: match on substrings."""
    import json
    import tempfile
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as td:  # the trace lists every kernel, also those launched outside torch operators
        path = os.path.join(td, "trace.json")
        prof.export_chrome_trace(path)
        events = json.load(open(path)).get("traceEvents", [])
    return res, {e.get("name", "") for e in events if e.get("cat") == "kernel"}


def assert_kernels(names, ran=(), not_ran=()):
    for k in ran:
        assert any(k in n for n in names), f"{k} did not run; kernels: {sorted(n for n in names if 'bqc::' in n)}"
    for k in not_ran:
        assert not any(k in n for n in names), f"{k} ran; kernels: {sorted(n for n in names if 'bqc::' in n)}"


# Quality bytes where the kernels' unsigned forms of the reference's signed-char tests change behaviour: Q20 of the
# triplet walk, the last ordinary cutoff (94 + 33 = 127), the sign flip of (char)(q + 33) at 95, and values far into
# the negative range.  Bytes stay <= 222: from 223 on (char)(q + 33) wraps in the reference's own arithmetic.
QUAL_EDGES = (19, 20, 93, 94, 95, 99, 100, 127, 128, 199, 200, 222)


def mutate_qual(records, offsets, share=0.5, seed=0):
    """Rewrite the QUAL bytes of about `share` of the records in place: per read either one edge value throughout (so a
    cutoff at that value sees whole windows), runs of edge values, or independent draws from 0..222 weighted towards
    the edges."""
    rng = np.random.default_rng(seed)
    edges = np.array(QUAL_EDGES, dtype=np.uint8)
    for i in range(len(offsets) - 1):
        if rng.random() >= share:
            continue
        o = int(offsets[i]) + 4
        l_name = int(records[o + 8])
        n_cig = int(records[o + 12]) | int(records[o + 13]) << 8
        l_seq = int(records[o + 16]) | int(records[o + 17]) << 8 | int(records[o + 18]) << 16
        qual = o + 32 + l_name + 4 * n_cig + (l_seq + 1) // 2
        mode = rng.integers(3)
        if mode == 0:
            q = np.full(l_seq, rng.choice(edges), dtype=np.uint8)
        elif mode == 1:
            q = np.repeat(rng.choice(edges, size=l_seq // 16 + 1), 16)[:l_seq]
        else:
            q = np.where(rng.random(l_seq) < 0.5, rng.choice(edges, size=l_seq), rng.integers(0, 223, size=l_seq)).astype(np.uint8)
        records[qual:qual + l_seq] = q


def against_oracle(tmp_path, stream, opts=("-c", "chr1,chr2"), expect_rc=0):
    """The drop-in command and the oracle on the same uncompressed BAM stream (golden genome): same exit status and,
    on success, the same .bamqc."""
    fasta = tmp_path / "g.fa"
    golden_genome().write_fasta(fasta)
    bam = tmp_path / "in.bam"
    bam.write_bytes(stream)
    o = subprocess.run([ensure_oracle(), "-r", str(fasta), "-o", str(tmp_path / "o.bamqc")] + list(opts) + [str(bam)], capture_output=True, text=True)
    g = run_cli(["-r", fasta, "-o", tmp_path / "g.bamqc"] + list(opts) + [bam])
    assert o.returncode == expect_rc, o.stderr
    assert g.returncode == expect_rc, g.stderr + g.stdout
    if expect_rc == 0:
        diffs = diff_bamqc(tmp_path / "o.bamqc", tmp_path / "g.bamqc")
        assert not diffs, "\n".join(diffs)
    return o, g


# ------------------------------------------------------------------------------------------------------
# hand-built BAM records for edge cases
# ------------------------------------------------------------------------------------------------------
import struct

NT16 = "=ACMGRSVTWYHKDBN"
CIGAR_OPS = "MIDNSHP=X"
GOLDEN = os.path.join(ROOT, "tests", "golden")
REF_BIN = os.path.join(ORACLE_DIR, "_ref", "bamqualcheck_ref")


def bam_record(name="r", flag=0x41, rid=0, pos=100, mapq=60, cigar=((150, "M"),), seq=None, qual=None, nrid=0, npos=300,
               tlen=350, tags=(("RG", "Z", "L1"), ("NM", "C", 0), ("AS", "C", 150))):
    """One inflated BAM record (block_size prefix included)."""
    seq = seq if seq is not None else "ACGT" * 37 + "AC"
    qual = qual if qual is not None else [30] * len(seq)
    b = bytearray()
    nm = name.encode() + b"\0"
    b += struct.pack("<iiBBHHHiiii", rid, pos, len(nm), mapq, 4680, len(cigar), flag, len(seq), nrid, npos, tlen)
    b += nm
    for n, op in cigar:
        b += struct.pack("<I", (n << 4) | CIGAR_OPS.index(op))
    codes = [NT16.index(c) for c in seq]
    for i in range(0, len(codes), 2):
        b.append((codes[i] << 4) | (codes[i + 1] if i + 1 < len(codes) else 0))
    b += bytes(qual)
    for key, ty, val in tags:
        b += key.encode() + ty.encode()
        if ty == "Z":
            b += val.encode() + b"\0"
        elif ty in "cC":
            b += struct.pack("<b" if ty == "c" else "<B", val)
        elif ty in "sS":
            b += struct.pack("<h" if ty == "s" else "<H", val)
        elif ty in "iI":
            b += struct.pack("<i" if ty == "i" else "<I", val)
        elif ty == "f":
            b += struct.pack("<f", val)
        elif ty == "A":
            b += val.encode()
        elif ty == "B":  # val = (subtype, [values])
            sub, vals = val
            b += sub.encode() + struct.pack("<i", len(vals)) + b"".join(struct.pack("<" + {"c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I", "f": "f"}[sub], v) for v in vals)
    return struct.pack("<i", len(b)) + bytes(b)


def bam_stream(records, refs=(("chr1", 60000), ("chr2", 40000), ("chrX", 20000)), lanes=("L1",), sample="S1"):
    """Uncompressed BAM byte stream: header + records."""
    text = "@HD\tVN:1.6\tSO:coordinate\n" + "".join(f"@SQ\tSN:{n}\tLN:{l}\n" for n, l in refs) + \
        "".join(f"@RG\tID:{l}\tSM:{sample}\n" for l in lanes)
    h = b"BAM\1" + struct.pack("<i", len(text)) + text.encode() + struct.pack("<i", len(refs))
    for n, l in refs:
        h += struct.pack("<i", len(n) + 1) + n.encode() + b"\0" + struct.pack("<i", l)
    return h + b"".join(records)


def golden_genome():
    from bamqc_b200 import synth
    return synth.Genome.make(77, ["chr1", "chr2", "chrX"], [60000, 40000, 20000])


def run_cli(args):
    """The product CLI (bamqc_b200/bin/bamqualcheck)."""
    exe = os.path.join(ROOT, "bamqc_b200", "bin", "bamqualcheck")
    return subprocess.run([exe] + [str(a) for a in args], capture_output=True, text=True)


def bgzf_block_starts(comp):
    """Offsets of the BGZF blocks in a compressed byte array (BSIZE from the BC extra field, SAM/BAM spec 4.1)."""
    b = bytes(comp)
    out, p = [], 0
    while p + 18 <= len(b):
        assert b[p:p + 4] == b"\x1f\x8b\x08\x04"
        xlen = struct.unpack_from("<H", b, p + 10)[0]
        x, bsize = p + 12, None
        while x + 4 <= p + 12 + xlen:
            slen = struct.unpack_from("<H", b, x + 2)[0]
            if b[x:x + 2] == b"BC" and slen == 2:
                bsize = struct.unpack_from("<H", b, x + 4)[0]
            x += 4 + slen
        out.append(p)
        p += bsize + 1
    return out


def bam_records_to_sam(stream_bytes):
    """SAM text (header + alignment lines) of an uncompressed BAM byte stream (SAM/BAM specification 4.2)."""
    b = bytes(stream_bytes)
    assert b[:4] == b"BAM\1"
    l_text = struct.unpack_from("<i", b, 4)[0]
    text = b[8:8 + l_text].decode()
    p = 8 + l_text
    n_ref = struct.unpack_from("<i", b, p)[0]
    p += 4
    names = []
    for _ in range(n_ref):
        l_name = struct.unpack_from("<i", b, p)[0]
        names.append(b[p + 4:p + 4 + l_name - 1].decode())
        p += 4 + l_name + 4
    lines = []
    while p + 4 <= len(b):
        bs = struct.unpack_from("<i", b, p)[0]
        r = b[p + 4:p + 4 + bs]
        p += 4 + bs
        rid, pos, l_name, mapq, _bin, n_cig, flag, l_seq, nrid, npos, tlen = struct.unpack_from("<iiBBHHHiiii", r, 0)
        q = 32
        name = r[q:q + l_name - 1].decode()
        q += l_name
        cig = ""
        for _ in range(n_cig):
            c = struct.unpack_from("<I", r, q)[0]
            cig += "%d%s" % (c >> 4, CIGAR_OPS[c & 15])
            q += 4
        seq = "".join(NT16[(r[q + i // 2] >> (4 if i % 2 == 0 else 0)) & 15] for i in range(l_seq))
        q += (l_seq + 1) // 2
        qual = "".join(chr(33 + x) for x in r[q:q + l_seq])
        q += l_seq
        tags = []
        while q + 3 <= len(r):
            key, ty = r[q:q + 2].decode(), chr(r[q + 2])
            q += 3
            if ty == "A":
                tags.append(f"{key}:A:{chr(r[q])}"); q += 1
            elif ty in "cCsSiI":
                fmt = {"c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I"}[ty]
                v = struct.unpack_from("<" + fmt, r, q)[0]
                tags.append(f"{key}:i:{v}"); q += struct.calcsize(fmt)
            elif ty == "f":
                tags.append(f"{key}:f:{struct.unpack_from('<f', r, q)[0]!r}"); q += 4
            elif ty in "ZH":
                e = r.index(b"\0", q)
                tags.append(f"{key}:{ty}:{r[q:e].decode()}"); q = e + 1
            elif ty == "B":
                sub = chr(r[q]); cnt = struct.unpack_from("<i", r, q + 1)[0]
                fmt = {"c": "b", "C": "B", "s": "h", "S": "H", "i": "i", "I": "I", "f": "f"}[sub]
                vals = struct.unpack_from("<%d%s" % (cnt, fmt), r, q + 5)
                tags.append(f"{key}:B:{sub}," + ",".join(repr(v) for v in vals)); q += 5 + cnt * struct.calcsize(fmt)
            else:
                raise ValueError(ty)
        rn = names[rid] if rid >= 0 else "*"
        nn = "*" if nrid < 0 else ("=" if nrid == rid else names[nrid])
        lines.append("\t".join([name, str(flag), rn, str(pos + 1), str(mapq), cig or "*", nn, str(npos + 1), str(tlen), seq or "*",
                                qual or "*"] + tags))
    return text + "\n".join(lines) + ("\n" if lines else "")
