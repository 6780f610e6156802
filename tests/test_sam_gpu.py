"""SAM text encoded on the device (bqc_submit_sam / bqc_sam_to_bam, kernel_sam.cuh) against the host encoder, the
same records as BAM, and the CPU oracle reading the same SAM text."""
import os
import subprocess

import numpy as np
import pytest

import bqc_testutil as util
from bamqc_b200 import BamQCError, Engine, synth

pytestmark = pytest.mark.gpu
EXE = os.path.join(util.ROOT, "bamqc_b200", "bin", "bamqualcheck")
B_LINE = b"bx\t99\tchr1\t100\t60\t4M\t=\t300\t350\tACGT\tIIII\tRG:Z:L1\tAS:i:3\tXB:B:S,1,2,3\n"


def _split(sam):
    lines = sam.encode().split(b"\n")
    head = b"".join(l + b"\n" for l in lines if l.startswith(b"@"))
    body = b"".join(l + b"\n" for l in lines if l and not l.startswith(b"@"))
    return head, body


def _library(tmp_path, seed=51, n_pairs=3000, stress=True, **kw):
    os.makedirs(tmp_path, exist_ok=True)
    genome = util.golden_genome()
    lib_ = synth.Library(seed=seed, n_pairs=n_pairs, **kw)
    if stress:
        lib_ = lib_.stress()
    records, offsets = synth.generate(genome, lib_)
    fasta, bam = tmp_path / "ref.fa", tmp_path / "in.ubam"
    genome.write_fasta(fasta)
    synth.write_bam(bam, genome, lib_, records, int(offsets[-1]))
    return genome, lib_, fasta, bam


def _clamp_qual(records, offsets, top=93):
    """Quality bytes above `top` lowered to it, so that the SAM text of the records stays ASCII (the device grammar)."""
    for k in range(len(offsets) - 1):
        o = int(offsets[k]) + 4
        l_name, n_cig, l_seq = int(records[o + 8]), int(records[o + 12]) | int(records[o + 13]) << 8, int(np.frombuffer(records[o + 16:o + 20], np.int32)[0])
        q = o + 32 + l_name + 4 * n_cig + (l_seq + 1) // 2
        seg = records[q:q + l_seq]
        if l_seq and seg[0] != 0xFF:
            np.minimum(seg, top, out=seg)


def _stress_ascii(tmp_path, seed=52):
    genome = util.golden_genome()
    lib_ = synth.Library(seed=seed, n_pairs=3000).stress()
    records, offsets = synth.generate(genome, lib_)
    _clamp_qual(records, offsets)
    os.makedirs(tmp_path, exist_ok=True)
    bam = tmp_path / "stress_ascii.ubam"
    synth.write_bam(bam, genome, lib_, records, int(offsets[-1]))
    return genome, lib_, bam


def test_device_records_equal_the_host_encoder(tmp_path):
    genome, lib_, fasta, bam = _library(tmp_path, stress=False)
    head, body = _split(util.bam_records_to_sam(open(bam, "rb").read()))
    _, _, _, sbam = _library(tmp_path / "s", seed=52)
    _, stress_body = _split(util.bam_records_to_sam(open(sbam, "rb").read()))
    _, _, abam = _stress_ascii(tmp_path / "a")
    _, ascii_body = _split(util.bam_records_to_sam(open(abam, "rb").read()))
    odd = [util.bam_record(name=f"s{i}", flag=0x63 if i % 2 == 0 else 0x93, pos=1000 + 3 * i, npos=1200, tlen=350,
                           tags=(("RG", "Z", "L1"), ("NM", "i", i * 977 - 30000), ("XF", "f", 1.5 + i), ("AS", "s", 120), ("XA", "A", "q")))
           for i in range(50)]
    _, odd_body = _split(util.bam_records_to_sam(util.bam_stream(odd)))
    edge = (b"e1\t0\tchr2\t-5\t255\t3S1M\t*\t0\t-2147483649\tacgtn.=X\t*\tXI:i:-2147483649\tXJ:i:4294967296\tXF:f:-0\n"
            b"e2\t65535\t=\t2147483648\t7\t*\tchrX\t1\t0\t*\t*\tXF:f:1e22\tXG:f:0.1\tXZ:Z:a b:c\tXH:H:0AFF\n"
            b"\r\n\n"
            b"e3\t1\tnochr\t1\t1\t1M\tchr1\t1\t1\tA\tII\tXA:A:\r\n")
    eng = Engine(lane_ids=synth.lane_ids(lib_), ref_names=genome.names)
    for text, fast in ((body, True), (odd_body, True), (edge, True), (ascii_body, True), (stress_body, False)):
        before = eng.sam_host_lines
        dev = eng.sam_to_bam(text)
        if fast:   # aligner-like text stays on the device (the stress library has quality bytes beyond ASCII)
            assert eng.sam_host_lines == before
        before = eng.sam_host_lines
        host = eng.sam_to_bam(text + B_LINE)   # a B array: the whole text goes through the host encoder
        assert eng.sam_host_lines > before
        assert host[:len(dev)] == dev
        assert len(host) > len(dev)
    # a final line without a newline counts when the text is complete
    assert eng.sam_to_bam(edge.rstrip(b"\r\n")) == eng.sam_to_bam(edge)
    eng.close()


def test_device_encodes_the_selftest_lines_like_the_host(tmp_path):
    """The random odd lines of tests/sam_selftest.cpp that its fast path accepts, through the device build of the
    grammar (its __CUDA_ARCH__ branches: __dmul_rn / __ddiv_rn / __double2float_rn / __float_as_uint) against the host
    encoder."""
    exe, lines = str(tmp_path / "sam_selftest"), tmp_path / "odd.sam"
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(util.ROOT, "tests", "sam_selftest.cpp")], check=True)
    r = subprocess.run([exe, "--emit", str(lines), "60000"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout
    text = open(lines, "rb").read()
    names = ["chr1", "chr2", "chr10", "chrX", "chr1", "c", "chr1_alt", "chr", "HLA-A*01:01", "chrM"]   # kNames of the self-test
    eng = Engine(lane_ids=("L1",), ref_names=names)
    dev = eng.sam_to_bam(text)
    assert eng.sam_host_lines == 0
    host = eng.sam_to_bam(text + B_LINE)
    assert eng.sam_host_lines > 0
    assert len(host) > len(dev) and host[:len(dev)] == dev
    assert text.count(b"\n") > 10000
    eng.close()


def test_submit_sam_equals_submit_stream(tmp_path):
    genome, lib_, fasta, bam = _library(tmp_path, seed=77, n_pairs=4000, stress=False, n_lanes=3)
    raw = open(bam, "rb").read()
    head, body = _split(util.bam_records_to_sam(raw))

    def run(feed):
        eng = Engine(lane_ids=synth.lane_ids(lib_), ref_names=genome.names, chroms="chr1,chr2", klist=(15, 32), qlist=(10, 17), staging_bytes=1 << 20)
        for rid, (p, n) in enumerate(zip(genome.packed, genome.lengths)):
            eng.set_reference(rid, p, n)
        feed(eng)
        eng.finish()
        return eng

    # the BAM side: the file's own records, after its header
    hdr_len = int(np.frombuffer(raw[4:8], dtype=np.int32)[0])
    p = 8 + hdr_len
    n_ref = int(np.frombuffer(raw[p:p + 4], dtype=np.int32)[0])
    p += 4
    for _ in range(n_ref):
        p += 4 + int(np.frombuffer(raw[p:p + 4], dtype=np.int32)[0]) + 4
    enc = raw[p:]

    def feed_stream(eng):
        for i in range(0, len(enc), 700_000):
            eng.submit_stream(enc[i:i + 700_000], last=i + 700_000 >= len(enc))

    rng = np.random.default_rng(5)
    cuts, a = [], 0
    while a < len(body):   # arbitrary line ends, every chunk within the 1 MB staging buffer
        c = body.rfind(b"\n", a, a + int(rng.integers(100, 900_000))) + 1
        a = c if c > a else body.index(b"\n", a) + 1
        cuts.append(a)

    def feed_sam(eng):
        a = 0
        for c in cuts:
            if c > a:
                eng.submit_sam(body[a:c], last=c == len(body))
            a = c

    e1, e2 = run(feed_stream), run(feed_sam)
    assert e2.sam_host_lines == 0
    for lane in range(3):
        for name, f in __import__("bamqc_b200").FIELDS.items():
            for sub in (0, 1) if name in ("AVGQUAL",) else (0,):
                try:
                    a = e1.table(f, lane=lane, sub=sub)
                except BamQCError:
                    continue
                assert np.array_equal(a, e2.table(f, lane=lane, sub=sub)), (lane, name)
        for qk in range(4):
            assert np.array_equal(e1.sketch(lane=lane, qk=qk), e2.sketch(lane=lane, qk=qk))
    e1.close()
    # a chunk that does not end at a line end is refused
    with pytest.raises(BamQCError) as ei:
        e2.reset()
        e2.submit_sam(body[:cuts[0] - 5])
    assert ei.value.code == 33
    e2.close()


def _cli(args, sam):
    return subprocess.run([EXE] + [str(a) for a in args] + ["-"], input=sam, capture_output=True)


def _oracle(args, sam):
    return subprocess.run([util.ensure_oracle()] + [str(a) for a in args] + ["-"], input=sam, capture_output=True)


@pytest.mark.parametrize("case", ["stress", "three_lanes_kq", "long_reads", "staging_1mb", "fallback_mid"])
def test_cli_stdin_against_bam_and_oracle(case, tmp_path):
    kw = dict(stress=case == "stress", seed=91)
    if case == "three_lanes_kq":
        kw["n_lanes"] = 3
    if case == "long_reads":
        kw.update(read_len=1500, ins_mean=3200.0, ins_min=3000, ins_max=3600, n_pairs=600)
    if case in ("staging_1mb", "fallback_mid"):
        kw["n_pairs"] = 12000
    if case == "stress":   # qualities clamped to ASCII so that the device encoder runs on the stress records
        genome, lib_, bam = _stress_ascii(tmp_path, seed=91)
        fasta = tmp_path / "ref.fa"
        genome.write_fasta(fasta)
    else:
        genome, lib_, fasta, bam = _library(tmp_path, **kw)
    opts = ["-r", fasta, "-c", "chr1,chr2"]
    if case == "three_lanes_kq":
        opts += ["-k", "15,32,63", "-q", "10,17"]
    if case in ("staging_1mb", "fallback_mid"):
        opts += ["--staging-mb", "1"]
    sam = util.bam_records_to_sam(open(bam, "rb").read()).encode()
    if case == "fallback_mid":   # one B array in the middle: that submission goes through the host encoder
        head, body = _split(sam.decode())
        mid = body.index(b"\n", len(body) // 2) + 1
        line = body[mid:body.index(b"\n", mid) + 1]
        sam = head + body[:mid] + line.rstrip(b"\n") + b"\tXB:B:c,1,-2\n" + body[body.index(b"\n", mid) + 1:]
    g1 = util.run_cli(opts + ["-o", tmp_path / "bam.bamqc", bam])
    assert g1.returncode == 0, g1.stderr
    g2 = _cli(opts + ["-o", tmp_path / "sam.bamqc", "--timing"], sam)
    assert g2.returncode == 0, g2.stderr
    timing = [l for l in g2.stderr.decode().splitlines() if l.startswith("BAMQC_TIMING")][0]
    host_lines = int(timing.split("sam_host_lines=")[1].split()[0])
    assert (host_lines > 0) == (case == "fallback_mid"), timing
    if case != "fallback_mid":
        assert not util.diff_bamqc(tmp_path / "bam.bamqc", tmp_path / "sam.bamqc")
    o = _oracle([x for x in opts if x not in ("--staging-mb", "1")] + ["-o", tmp_path / "oracle.bamqc"], sam)
    assert o.returncode == 0, o.stderr
    diffs = util.diff_bamqc(tmp_path / "oracle.bamqc", tmp_path / "sam.bamqc")
    assert not diffs, "\n".join(diffs)


def test_cli_minimal_lines_at_small_staging(tmp_path):
    """The shortest lines over many 1 MB submissions.  22-byte lines (the worst-case expansion the slot is sized for)
    carry no RG tag, which the reference and the oracle refuse: they are counted on the device and refused the same
    way.  31-byte lines with a mate flag and RG:Z:L1 (about the shortest the reference accepts) give the oracle's .bamqc."""
    genome = util.golden_genome()
    fasta = tmp_path / "ref.fa"
    genome.write_fasta(fasta)
    head = b"@SQ\tSN:chr1\tLN:60000\n@RG\tID:L1\tSM:S1\n"
    opts = ["-r", fasta, "-c", "chr1"]
    for line, ok in ((b"r\t4\t*\t0\t0\t*\t*\t0\t0\tA\tI\n", False), (b"r\t77\t*\t0\t0\t*\t*\t0\t0\tA\tI\tRG:Z:L1\n", True)):
        assert len(line) == (31 if ok else 22)
        sam = head + line * 150000
        g = _cli(opts + ["--staging-mb", "1", "-o", tmp_path / "sam.bamqc", "--timing"], sam)
        o = _oracle(opts + ["-o", tmp_path / "oracle.bamqc"], sam)
        assert g.returncode == o.returncode == (0 if ok else 1), (g.stderr, o.stderr)
        timing = [l for l in g.stderr.decode().splitlines() if l.startswith("BAMQC_TIMING")][0]
        assert "sam_host_lines=0" in timing, timing
        if ok:
            assert "records=150000 " in timing, timing
            diffs = util.diff_bamqc(tmp_path / "oracle.bamqc", tmp_path / "sam.bamqc")
            assert not diffs, "\n".join(diffs)


@pytest.mark.parametrize("case", ["malformed_k", "mate_flag_then_malformed", "rg_not_z", "missing_as"])
def test_cli_stdin_errors_match_the_oracle(case, tmp_path):
    genome = util.golden_genome()
    fasta = tmp_path / "ref.fa"
    genome.write_fasta(fasta)
    recs = [util.bam_record(name=f"s{i}", flag=0x63 if i % 2 == 0 else 0x93, pos=1000 + 3 * i, npos=1200, tlen=350,
                            tags=(("RG", "Z", "L1"), ("AS", "i", 100))) for i in range(400)]
    if case == "mate_flag_then_malformed":
        recs[100] = util.bam_record(name="nomate", flag=0x1, pos=2000, tags=(("RG", "Z", "L1"), ("AS", "i", 100)))
    if case == "rg_not_z":
        recs[150] = util.bam_record(name="rg", flag=0x63, pos=2000, tags=(("RG", "A", "L"), ("AS", "i", 100)))
    if case == "missing_as":
        recs[150] = util.bam_record(name="noas", flag=0x63, pos=2000, tags=(("RG", "Z", "L1"),))
    sam = util.bam_records_to_sam(util.bam_stream(recs)).encode()
    if case in ("malformed_k", "mate_flag_then_malformed"):
        head, body = _split(sam.decode())
        lines = body.split(b"\n")
        lines[300] = b"broken\t0\tchr1"
        sam = head + b"\n".join(lines)
    opts = ["-r", fasta, "-c", "chr1,chr2"]
    g = _cli(opts + ["-o", tmp_path / "g.bamqc"], sam)
    o = _oracle(opts + ["-o", tmp_path / "o.bamqc"], sam)
    assert g.returncode == o.returncode, (g.stderr, o.stderr)
    assert o.returncode != 0 or case == "missing_as"
    assert g.stdout == o.stdout
    # the oracle's SAM reader refuses a malformed line before it counts anything ("Could not open - for reading"); the
    # command keeps its message for it, and a fatal record in front of the malformed line is reported first
    expect = {"malformed_k": "ERROR: Could not read record from BAM File -",
              "mate_flag_then_malformed": "ERROR: No first or second flag in read in:  -"}
    if case in expect:
        assert [l for l in g.stderr.decode().splitlines() if l.startswith("ERROR")] == [expect[case]], g.stderr
    g_out = tmp_path / "g.bamqc"
    if o.returncode:
        assert not g_out.exists() or g_out.stat().st_size == 0
    else:
        assert not util.diff_bamqc(tmp_path / "o.bamqc", g_out)


def test_sam_kernels_run(tmp_path):
    genome, lib_, fasta, bam = _library(tmp_path, stress=False, n_pairs=2000)
    head, body = _split(util.bam_records_to_sam(open(bam, "rb").read()))

    def go():
        eng = Engine(lane_ids=synth.lane_ids(lib_), ref_names=genome.names)
        for rid, (p, n) in enumerate(zip(genome.packed, genome.lengths)):
            eng.set_reference(rid, p, n)
        eng.profile_enable(True)
        eng.submit_sam(body, last=True)
        eng.finish()
        prof = eng.profile_read()
        eng.close()
        return prof

    prof, names = util.kernel_names(go)
    util.assert_kernels(names, ran=("k_sam_nl_count", "k_sam_size", "k_sam_encode", "k_stats"), not_ran=("k_frame_speculate",))
    assert prof["k_sam"][1] == 1
