"""The drop-in command (bamqc_b200/bin/bamqualcheck: BGZF inflate on host threads -> pinned staging -> CUDA
engine through the C ABI -> .bamqc writer) against the committed golden outputs of the reference's own code,
and edge cases against the oracle."""
import os
import random
import subprocess

import numpy as np
import pytest

import bqc_testutil as util

pytestmark = pytest.mark.gpu
GOLD = util.GOLDEN
CASES = {
    "standard": ["-c", "chr1,chr2"],
    "stress": ["-c", "chr1,chr2"],
    "two_lanes_kq": ["-c", "chr1,chr2", "-k", "15,32,63", "-q", "10,17"],
    "long_insert": ["-c", "chr1,chr2,chrX", "-i", "3000", "-s", "7"],
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_cli_reproduces_reference_bamqc(case, tmp_path):
    out = tmp_path / "gpu.bamqc"
    r = util.run_cli(["-r", os.path.join(GOLD, "genome.fa"), "-o", out] + CASES[case] + [os.path.join(GOLD, case + ".bam")])
    assert r.returncode == 0, r.stderr + r.stdout
    diffs = util.diff_bamqc(os.path.join(GOLD, case + ".bamqc"), out)
    assert not diffs, "\n".join(diffs)


_against_oracle = util.against_oracle


def test_empty_input(tmp_path):
    """Header only: every lane still flushes two empty coverage windows (src/bamqualcheck.cpp:447-453)."""
    _against_oracle(tmp_path, util.bam_stream([]))
    line = [l for l in open(tmp_path / "g.bamqc") if l.startswith("genome_coverage_histogram")][0].split()
    assert line[1] == "2000"


def test_ragged_lengths_iupac_and_odd_tags(tmp_path):
    rng = random.Random(3)
    genome = util.golden_genome()
    recs = []
    pos = 500
    for i in range(400):
        L = rng.choice([32, 33, 50, 75, 100, 101, 149, 150, 151, 200, 250])
        pos += rng.randint(1, 120)
        start = pos
        ref = "".join("ACGT"[(int(genome.packed[0][(start + j) // 4]) >> (2 * ((start + j) % 4))) & 3] for j in range(L))
        seq = list(ref)
        for j in range(L):
            x = rng.random()
            if x < 0.01:
                seq[j] = rng.choice("MRWSYKVHDBN=")  # IUPAC codes exercise the non-ACGT paths
            elif x < 0.03:
                seq[j] = rng.choice("ACGT")
        qual = [rng.choice([2, 12, 23, 37, 41, 60, 93]) for _ in range(L)]
        rev = rng.random() < 0.5
        first = rng.random() < 0.5
        flag = 0x1 | 0x2 | (0x10 if rev else 0x20) | (0x40 if first else 0x80)
        if rng.random() < 0.05:
            flag |= 0x400
        nm_type = rng.choice(["c", "C", "s", "S", "i", "I"])
        tags = [("XA", "Z", "junk"), ("RG", "Z", "L1"), ("XB", "B", ("S", [1, 2, 3])), ("NM", nm_type, rng.randint(0, 5)),
                ("XF", "f", 1.5), ("AS", rng.choice(["C", "s", "i"]), rng.randint(40, 150)), ("XH", "H", "1AE3")]
        if rng.random() < 0.1:
            tags.append(("NM", "C", 2))  # a second NM is counted again by the reference (no break in the loop)
        recs.append(util.bam_record(name=f"q{i}", flag=flag, rid=0, pos=start, mapq=rng.choice([0, 30, 59, 60]),
                                    cigar=((L, "M"),), seq="".join(seq), qual=qual, nrid=0, npos=start + 200,
                                    tlen=rng.choice([-1, 1]) * rng.randint(0, 1500), tags=tuple(tags)))
    _against_oracle(tmp_path, util.bam_stream(recs))


@pytest.mark.parametrize("name,bad", [
    ("rg_type", dict(flag=0x63, tags=(("RG", "i", 5), ("NM", "C", 0), ("AS", "C", 150)))),
    ("no_mate_flag", dict(flag=0x1, tags=(("RG", "Z", "L1"), ("NM", "C", 0), ("AS", "C", 150)))),
    ("no_as", dict(flag=0x63, tags=(("RG", "Z", "L1"), ("NM", "C", 0)))),
    ("negative_as", dict(flag=0x63, tags=(("RG", "Z", "L1"), ("NM", "C", 0), ("AS", "c", -3)))),
])
def test_fatal_conditions_exit_1(tmp_path, name, bad):
    good = util.bam_record(name="a", flag=0x63, pos=1000, npos=1200, tlen=350)
    o, g = _against_oracle(tmp_path, util.bam_stream([good, util.bam_record(name="b", pos=1100, **bad), good]), opts=("-c", "chr1"), expect_rc=1)
    if name == "rg_type":
        assert "Read does not have Z" in g.stdout
    if name == "no_mate_flag":
        assert "No first or second flag" in g.stderr


def test_cli_argument_errors(tmp_path):
    assert util.run_cli(["-o", tmp_path / "x", os.path.join(GOLD, "standard.bam")]).returncode == 1          # -r is required
    assert util.run_cli(["-r", os.path.join(GOLD, "genome.fa"), os.path.join(GOLD, "standard.bam")]).returncode == 1  # -o is required
    r = util.run_cli(["-r", os.path.join(GOLD, "genome.fa"), "-o", tmp_path / "x", tmp_path / "missing.bam"])
    assert r.returncode == 1 and "Could not open" in r.stderr
    assert util.run_cli(["--help"]).returncode == 0


def test_multi_batch_streaming_with_small_staging(tmp_path):
    """Many tiny staging buffers: records straddling BGZF blocks and buffer boundaries are carried over."""
    from bamqc_b200 import Engine, synth
    genome = util.golden_genome()
    lib_ = synth.Library(seed=31, n_pairs=4000)
    records, offsets = synth.generate(genome, lib_)
    fasta, bam = tmp_path / "g.fa", tmp_path / "in.ubam"
    genome.write_fasta(fasta)
    synth.write_bam(bam, genome, lib_, records, int(offsets[-1]))
    r = util.run_oracle(bam, fasta, tmp_path / "o.bamqc", chroms="chr1,chr2")
    assert r.returncode == 0
    eng = Engine(lane_ids=["L1"], ref_names=genome.names, chroms="chr1,chr2", staging_bytes=64 << 10)
    for rid, (p, n) in enumerate(zip(genome.packed, genome.lengths)):
        eng.set_reference(rid, p, n)
    n_bytes = int(offsets[-1])
    pos = 0
    carry = np.zeros(0, dtype=np.uint8)
    while pos < n_bytes:
        buf = eng.acquire_staging()
        take = min(buf.size - carry.size, n_bytes - pos, 50000)
        buf[:carry.size] = carry
        buf[carry.size:carry.size + take] = records[pos:pos + take]
        filled = carry.size + take
        pos += take
        offs = np.zeros(filled // 36 + 2, dtype=np.uint64)
        n = eng.lib.bqc_frame_records(buf.ctypes.data, filled, offs.ctypes.data, offs.size)
        whole = int(offs[n])
        carry = buf[whole:filled].copy()
        if n:
            eng.submit(buf, offs[:n + 1], n_bytes=whole)
    assert carry.size == 0
    eng.finish()
    eng.write_bamqc("S1", tmp_path / "g.bamqc")
    eng.close()
    diffs = util.diff_bamqc(tmp_path / "o.bamqc", tmp_path / "g.bamqc")
    assert not diffs, "\n".join(diffs)


def test_homopolymer_reads_overflow_the_16_bit_eightmer_counters(tmp_path):
    """k_eightmer keeps 16-bit counters in shared memory: poly-A / poly-T / poly-C reads push single bins far past
    65535 inside one CTA (wrap of a low field with its carry into the neighbour, wrap of a high field), and the
    low-quality stretches exercise the queued sketch probes."""
    recs = []
    pos = 100
    for i in range(1800):
        base = "ATC"[i % 3]
        pos += 7
        qual = [37] * 150
        if i % 5 == 0:
            qual[40] = 2
        flag = 0x1 | 0x2 | (0x10 if i % 4 == 1 else 0x20) | (0x40 if i % 2 == 0 else 0x80)
        recs.append(util.bam_record(name=f"h{i}", flag=flag, rid=0, pos=pos, mapq=60, cigar=((150, "M"),), seq=base * 150, qual=qual,
                                    nrid=0, npos=pos + 200, tlen=350 if i % 2 == 0 else -350))
    _against_oracle(tmp_path, util.bam_stream(recs))


def test_sam_on_stdin_gives_the_same_bamqc_as_the_bam_file(tmp_path):
    """`bamqualcheck ... -` (src/bamqualcheck.cpp:252-260): the same records as SAM text on stdin."""
    import subprocess
    from bamqc_b200 import synth
    genome = util.golden_genome()
    lib_ = synth.Library(seed=51, n_pairs=3000).stress()
    records, offsets = synth.generate(genome, lib_)
    fasta, bam = tmp_path / "ref.fa", tmp_path / "in.ubam"
    genome.write_fasta(fasta)
    synth.write_bam(bam, genome, lib_, records, int(offsets[-1]))
    g1 = util.run_cli(["-r", fasta, "-c", "chr1,chr2", "-o", tmp_path / "bam.bamqc", bam])
    assert g1.returncode == 0, g1.stderr
    sam = util.bam_records_to_sam(open(bam, "rb").read())
    exe = os.path.join(util.ROOT, "bamqc_b200", "bin", "bamqualcheck")
    g2 = subprocess.run([exe, "-r", str(fasta), "-c", "chr1,chr2", "-o", str(tmp_path / "sam.bamqc"), "-"], input=sam, capture_output=True, text=True)
    assert g2.returncode == 0, g2.stderr
    assert "Reading from stdin" in g2.stderr
    diffs = util.diff_bamqc(tmp_path / "bam.bamqc", tmp_path / "sam.bamqc")
    assert not diffs, "\n".join(diffs)
    # ... and as the CPU oracle reading the same SAM text with its own, independent SAM reader (oracle/bamqc_oracle.cpp: samToBam)
    o = subprocess.run([util.ensure_oracle(), "-r", str(fasta), "-c", "chr1,chr2", "-o", str(tmp_path / "oracle_sam.bamqc"), "-"], input=sam, capture_output=True, text=True)
    assert o.returncode == 0, o.stderr
    diffs = util.diff_bamqc(tmp_path / "oracle_sam.bamqc", tmp_path / "sam.bamqc")
    assert not diffs, "\n".join(diffs)
    # the odd tag types of the hand-made records survive the text round trip too
    recs = [util.bam_record(name=f"s{i}", flag=0x63 if i % 2 == 0 else 0x93, pos=1000 + 3 * i, npos=1200, tlen=350,
                            tags=(("RG", "Z", "L1"), ("XB", "B", ("S", [1, 2, 3])), ("NM", "i", i % 4), ("XF", "f", 1.5), ("AS", "s", 120), ("XA", "A", "q")))
            for i in range(50)]
    stream = util.bam_stream(recs)
    open(tmp_path / "h.ubam", "wb").write(stream)
    g3 = util.run_cli(["-r", fasta, "-c", "chr1", "-o", tmp_path / "h_bam.bamqc", tmp_path / "h.ubam"])
    g4 = subprocess.run([exe, "-r", str(fasta), "-c", "chr1", "-o", str(tmp_path / "h_sam.bamqc"), "-"], input=util.bam_records_to_sam(stream),
                        capture_output=True, text=True)
    assert g3.returncode == 0 and g4.returncode == 0, g3.stderr + g4.stderr
    assert not util.diff_bamqc(tmp_path / "h_bam.bamqc", tmp_path / "h_sam.bamqc")
    o2 = subprocess.run([util.ensure_oracle(), "-r", str(fasta), "-c", "chr1", "-o", str(tmp_path / "h_oracle.bamqc"), "-"], input=util.bam_records_to_sam(stream),
                        capture_output=True, text=True)
    assert o2.returncode == 0, o2.stderr
    assert not util.diff_bamqc(tmp_path / "h_oracle.bamqc", tmp_path / "h_sam.bamqc")


def test_large_deletions(tmp_path):
    """Summed deletion lengths up to 4095 bp in one read: the reference resizes `deletions` to the largest value seen
    (src/QualityCheck.hpp:261-265) and the engine's histogram has 4096 bins.  (Reads like these run past the reference's
    two coverage windows, where src/OverallNumbers.hpp:126-129 writes outside `v2`; the oracle and the engine drop those
    writes, the reference's own code aborts in free() -- so the oracle is the checker here.)  From 4096 bp on the engine
    reports BQC_ERR_UNSUPPORTED."""
    genome = util.golden_genome()
    fasta = tmp_path / "ref.fa"
    genome.write_fasta(fasta)

    def records(dels):
        recs = []
        for i, dl in enumerate(dels):
            recs.append(util.bam_record(name=f"d{i}", flag=0x63 if i % 2 == 0 else 0x93, pos=1000 + 40 * i, npos=1400, tlen=500,
                                        cigar=((50, "M"), (dl, "D"), (100, "M")),
                                        tags=(("RG", "Z", "L1"), ("NM", "i", dl + (i % 3)), ("AS", "C", 140))))
        return recs

    recs = records((3, 2000, 4095, 7))
    recs.append(util.bam_record(name="dd", flag=0x63, pos=1300, npos=1500, tlen=400, cigar=((30, "M"), (2000, "D"), (60, "M"), (2000, "D"), (60, "M")),
                                tags=(("RG", "Z", "L1"), ("NM", "i", 4000), ("AS", "C", 140))))   # two deletions in one read add up
    open(tmp_path / "d.ubam", "wb").write(util.bam_stream(recs))
    o = util.run_oracle(tmp_path / "d.ubam", fasta, tmp_path / "oracle.bamqc", chroms="chr1")
    assert o.returncode == 0, o.stderr
    g = util.run_cli(["-r", fasta, "-c", "chr1", "-o", tmp_path / "gpu.bamqc", tmp_path / "d.ubam"])
    assert g.returncode == 0, g.stderr
    diffs = util.diff_bamqc(tmp_path / "oracle.bamqc", tmp_path / "gpu.bamqc")
    assert not diffs, "\n".join(diffs)
    open(tmp_path / "e.ubam", "wb").write(util.bam_stream(records((3, 4096))))
    g = util.run_cli(["-r", fasta, "-c", "chr1", "-o", tmp_path / "e.bamqc", tmp_path / "e.ubam"])
    assert g.returncode != 0 and "capacit" in g.stderr


def test_records_larger_than_a_framing_window(tmp_path):
    """Records of 6-20 KB (long aux arrays) between ordinary ones: speculation windows of 4 KiB without any record
    start, chains that jump over several windows, through the raw-stream and the BGZF paths of the CLI."""
    rng = random.Random(5)
    recs = []
    pos = 300
    for i in range(600):
        pos += rng.randint(1, 40)
        big = rng.random() < 0.3
        tags = [("RG", "Z", "L1"), ("NM", "C", rng.randint(0, 3)), ("AS", "C", 140)]
        if big:
            tags.insert(1, ("XK", "B", ("S", [rng.randint(0, 65535) for _ in range(rng.choice([3000, 5000, 10000]))])))
        flag = 0x1 | 0x2 | (0x10 if i % 2 else 0x20) | (0x40 if i % 2 == 0 else 0x80)
        recs.append(util.bam_record(name=f"b{i}", flag=flag, rid=0, pos=pos, mapq=60, nrid=0, npos=pos + 100, tlen=250 if i % 2 == 0 else -250,
                                    tags=tuple(tags)))
    stream = util.bam_stream(recs)
    _against_oracle(tmp_path, stream)
    # the same file BGZF-compressed: device inflate + device framing
    from bamqc_b200 import synth
    comp = synth.bgzf_compress(np.frombuffer(stream, dtype=np.uint8), level=6)
    open(tmp_path / "in.bam", "wb").write(comp.tobytes())
    fasta = tmp_path / "ref2.fa"
    util.golden_genome().write_fasta(fasta)
    g = util.run_cli(["-r", fasta, "-c", "chr1,chr2", "-o", tmp_path / "g2.bamqc", tmp_path / "in.bam"])
    assert g.returncode == 0, g.stderr
    assert not util.diff_bamqc(tmp_path / "g.bamqc", tmp_path / "g2.bamqc")


# ---- streaming file input and several devices (the file is cut into one contiguous piece per engine) -----------------
@pytest.fixture(scope="module")
def big_bgzf(tmp_path_factory):
    """~600 k records as a level-1 BGZF BAM (~60 MB of file) + FASTA + the oracle's .bamqc."""
    from bamqc_b200 import synth
    d = tmp_path_factory.mktemp("big")
    genome = util.small_genome(seed=41, lengths=(3000000, 1500000, 200000))
    lib_ = synth.Library(seed=4100, n_pairs=300000)
    records, offsets = synth.generate(genome, lib_)
    fasta, bam = d / "g.fa", d / "big.bam"
    genome.write_fasta(fasta)
    synth.write_bam(bam, genome, lib_, records, int(offsets[-1]), level=1)
    r = util.run_oracle(bam, fasta, d / "oracle.bamqc", chroms="chr1,chr2")
    assert r.returncode == 0, r.stderr
    return d


@pytest.mark.parametrize("opts", [["--staging-mb", "8"], ["--devices", "0,0", "--staging-mb", "32"], ["--devices", "0,0,0", "--staging-mb", "16"]],
                         ids=["one_device_small_staging", "two_pieces", "three_pieces"])
def test_cli_streams_the_file_and_cuts_it_across_devices(big_bgzf, tmp_path, opts):
    """The command never holds the whole file: it reads staging-sized pieces (8 MB here: dozens of submissions with
    carried partial BGZF blocks).  With --devices the file is cut at BGZF block boundaries found by signature; the
    engines of the later pieces find their first record boundary themselves, the piece before completes its last
    record from the next piece's first bytes, and the coverage windows are resolved across the cuts.  Two or three
    engines share GPU 0 here; the output must be byte-identical to the oracle's on the whole file."""
    d = big_bgzf
    out = tmp_path / "gpu.bamqc"
    r = util.run_cli(["-r", d / "g.fa", "-c", "chr1,chr2", "-o", out, "--timing"] + opts + [d / "big.bam"])
    assert r.returncode == 0, r.stderr + r.stdout
    assert "could not be cut" not in r.stderr
    if "--devices" in opts:
        assert "devices=%d" % len(opts[1].split(",")) in r.stderr, r.stderr
    diffs = util.diff_bamqc(d / "oracle.bamqc", out)
    assert not diffs, "\n".join(diffs)


def test_cli_reads_bgzf_from_a_pipe(big_bgzf, tmp_path):
    d = big_bgzf
    out = tmp_path / "gpu.bamqc"
    exe = os.path.join(util.ROOT, "bamqc_b200", "bin", "bamqualcheck")
    with open(d / "big.bam", "rb") as f:
        p1 = subprocess.Popen(["cat"], stdin=f, stdout=subprocess.PIPE)
        r = subprocess.run([exe, "-r", str(d / "g.fa"), "-c", "chr1,chr2", "-o", str(out), "--staging-mb", "16", "/dev/stdin"], stdin=p1.stdout, capture_output=True, text=True)
        p1.wait()
    assert r.returncode == 0, r.stderr + r.stdout
    diffs = util.diff_bamqc(d / "oracle.bamqc", out)
    assert not diffs, "\n".join(diffs)
