"""The CPU oracle (oracle/bamqc_oracle.cpp, test infrastructure) against the committed golden fixtures that
were produced by the reference's own code (tests/golden/make_golden.py), and -- when oracle/_ref has been
built in this checkout -- against that reference build live on fresh seeds."""
import ctypes
import json
import os
import subprocess

import numpy as np
import pytest

import bqc_testutil as util

GOLD = util.GOLDEN
CASES = {
    "standard": ["-c", "chr1,chr2"],
    "stress": ["-c", "chr1,chr2"],
    "two_lanes_kq": ["-c", "chr1,chr2", "-k", "15,32,63", "-q", "10,17"],
    "long_insert": ["-c", "chr1,chr2,chrX", "-i", "3000", "-s", "7"],
}


@pytest.fixture(scope="module")
def olib():
    util.ensure_oracle()
    lib = ctypes.CDLL(os.path.join(util.ORACLE_DIR, "libbamqc_oracle.so"))
    return lib


@pytest.mark.parametrize("case", sorted(CASES))
def test_oracle_reproduces_reference_bamqc(case, tmp_path, oracle_bin):
    out = tmp_path / "o.bamqc"
    r = subprocess.run([oracle_bin, "-r", os.path.join(GOLD, "genome.fa"), "-o", str(out)] + CASES[case] +
                       [os.path.join(GOLD, case + ".bam")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    diffs = util.diff_bamqc(os.path.join(GOLD, case + ".bamqc"), out)
    assert not diffs, "\n".join(diffs)


@pytest.mark.parametrize("case", ["stress", "two_lanes_kq"])
def test_oracle_sam_reader_reproduces_reference_bamqc(case, tmp_path, oracle_bin):
    """The oracle's own SAM reader (samToBam; `bamqualcheck ... -`, src/bamqualcheck.cpp:252-260): the golden BAM as SAM
    text on stdin gives the golden .bamqc that the reference's code wrote for the BAM file."""
    import zlib
    raw = bytearray()
    b = open(os.path.join(GOLD, case + ".bam"), "rb").read()
    for p in util.bgzf_block_starts(b):
        xlen = int.from_bytes(b[p + 10:p + 12], "little")
        bsize = int.from_bytes(b[p + 16:p + 18], "little") + 1
        raw += zlib.decompress(b[p + 12 + xlen:p + bsize - 8], -15)
    sam = util.bam_records_to_sam(bytes(raw))
    out = tmp_path / "o.bamqc"
    r = subprocess.run([oracle_bin, "-r", os.path.join(GOLD, "genome.fa"), "-o", str(out)] + CASES[case] + ["-"], input=sam, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert "Reading from stdin" in r.stderr
    diffs = util.diff_bamqc(os.path.join(GOLD, case + ".bamqc"), out)
    assert not diffs, "\n".join(diffs)


def test_bamqc_shape():
    """80 lines per lane at defaults (SURVEY Appendix B)."""
    lines = open(os.path.join(GOLD, "standard.bamqc")).read().strip().split("\n")
    assert len(lines) == 80
    assert lines[0] == "sample_id S1" and lines[1] == "lane L1"
    keys = [l.split(" ")[0] for l in lines]
    assert keys[15] == "genome_coverage_histogram" and len(lines[15].split(" ")) == 102
    assert keys[16] == "insert_size_histogram" and len(lines[16].split(" ")) == 1002
    assert keys[59] == "8mer_count" and len(lines[59].split(" ")) == 65537
    assert keys[60:64] == ["32mer_count_after_qual_clipping_17", "distinct_32mer_count_after_qual_clipping_17",
                           "unique_32mer_count_after_qual_clipping_17", "32mer_F2_after_qual_clipping_17"]
    assert all(k.startswith("triplet_counts_") for k in keys[64:80])


def test_kmerstream_golden_vectors(olib):
    g = json.load(open(os.path.join(GOLD, "kmerstream_golden.json")))
    u64p = ctypes.POINTER(ctypes.c_uint64)
    hv = np.zeros(64, dtype=np.uint64)
    olib.oracle_rephash_hvals(1, hv.ctypes.data_as(u64p))
    assert ["%016x" % x for x in hv] == g["hvals_seed1"]
    # SURVEY Appendix D.1 / D.2 (vectors obtained from the reference's kmerstream sources during the survey)
    assert g["hvals_seed1"][2:4] == ["00077eff20ccc389", "4d65aacbffc11e85"]      # hvals[1] ('A')
    assert g["hvals_seed1"][40:42] == ["fd26000fa91f6c40", "bf87c8c44c6a3019"]    # hvals[20] ('T')
    assert g["windows"]["1:32"][:3] == ["dc73131adaf80128", "f125a4842f1d1742", "112077ce7e3ad4d5"]
    seq = g["seq42"].encode()
    for key, want in g["windows"].items():
        seed, k = map(int, key.split(":"))
        out = np.zeros(64, dtype=np.uint64)
        n = olib.oracle_rephash_windows(seed, k, seq, len(seq), out.ctypes.data_as(u64p))
        assert ["%016x" % x for x in out[:n]] == want, key
    olib.oracle_bitscan.restype = ctypes.c_uint64
    olib.oracle_bitscan.argtypes = [ctypes.c_uint64]
    for v, want in g["bitscan"].items():
        assert olib.oracle_bitscan(int(v)) == want
    assert g["bitscan"]["0"] == 63 and g["bitscan"]["8"] == 3


def test_streamcounter_and_hasher_golden(olib):
    import random
    import sys
    sys.path.insert(0, GOLD)
    import make_golden
    g = json.load(open(os.path.join(GOLD, "kmerstream_golden.json")))
    u64p = ctypes.POINTER(ctypes.c_uint64)
    olib.oracle_streamcounter.argtypes = [ctypes.c_double, ctypes.c_int, u64p, ctypes.c_uint64, u64p, u64p, u64p]
    for n_s, want in g["streamcounter"].items():
        n = int(n_s)
        rng = random.Random(42 + n)
        h = np.array([rng.getrandbits(64) for _ in range(n)] + [0] * (1 if n else 0), dtype=np.uint64)
        if n:
            h[::3] = h[0]
        out = np.zeros(6, dtype=np.uint64)
        olib.oracle_streamcounter(0.01, 1, h.ctypes.data_as(u64p), len(h), out.ctypes.data_as(u64p), None, None)
        assert [int(x) for x in out] == want, n
    assert g["streamcounter"]["0"][1:4] == [9223372036854775808, 9223372036854775808, 0]  # empty sketch (D.3)
    assert g["streamcounter"]["0"][4:6] == [32768, 32768]                                  # geometry (D.3)
    olib.oracle_hasher.argtypes = [ctypes.c_double, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_char_p, ctypes.c_char_p,
                                   ctypes.POINTER(ctypes.c_int), ctypes.c_int, u64p, u64p, u64p]
    for key, want in g["hasher"].items():
        q, k = map(int, key.split(":"))
        seqs, quals, lens = make_golden.hasher_reads(5)
        la = (ctypes.c_int * len(lens))(*lens)
        out = np.zeros(4, dtype=np.uint64)
        olib.oracle_hasher(0.01, 1, q, k, seqs, quals, la, len(lens), out.ctypes.data_as(u64p), None, None)
        assert [int(x) for x in out] == want, key
    assert g["hasher_fixed_read_sumcount"] == 14  # SURVEY D.4


needs_ref = pytest.mark.skipif(not os.path.exists(util.REF_BIN),
                               reason="oracle/_ref not built (make -C oracle ref REF=<BamQC source tree>)")


@needs_ref
@pytest.mark.parametrize("seed,kind", [(201, "standard"), (202, "stress"), (203, "sparse"), (204, "lanes"), (205, "short")])
def test_oracle_vs_reference_build_live(seed, kind, tmp_path, oracle_bin):
    from bamqc_b200 import synth
    lengths = (60000, 40000, 20000) if kind != "sparse" else (2500000, 1500000, 300000)
    genome = synth.Genome.make(seed, ["chr1", "chr2", "chrX"], list(lengths))
    lib_ = synth.Library(seed=seed, n_pairs=1500 if kind != "sparse" else 3000, n_lanes=3 if kind == "lanes" else 1,
                         read_len=76 if kind == "short" else 150, ins_mean=250 if kind == "short" else 400)
    if kind == "stress":
        lib_.stress()
    records, offsets = synth.generate(genome, lib_)
    fasta, bam = tmp_path / "g.fa", tmp_path / "in.bam"
    genome.write_fasta(fasta)
    synth.write_bam(bam, genome, lib_, records, int(offsets[-1]), level=1)
    opts = ["-c", "chr1,chr2"]
    a = subprocess.run([util.REF_BIN, "-r", str(fasta), "-o", str(tmp_path / "ref.bamqc")] + opts + [str(bam)], capture_output=True, text=True)
    b = subprocess.run([oracle_bin, "-r", str(fasta), "-o", str(tmp_path / "ora.bamqc")] + opts + [str(bam)], capture_output=True, text=True)
    assert a.returncode == 0 and b.returncode == 0, (a.stderr, b.stderr)
    diffs = util.diff_bamqc(tmp_path / "ref.bamqc", tmp_path / "ora.bamqc")
    assert not diffs, "\n".join(diffs)


def test_error_paths_match_reference_build(tmp_path, oracle_bin):
    """Fatal conditions of the reference: exit status 1 for RG of the wrong type, a read without first/last flag,
    and a triplet-eligible read without AS (src/bamqualcheck.cpp:81-97,385-389; src/TripletCounting.hpp:116-127).
    The oracle is held to the reference's recorded status on every checkout; the reference build is run as well
    where oracle/_ref has been built."""
    exes = [oracle_bin] + ([util.REF_BIN] if os.path.exists(util.REF_BIN) else [])
    util.golden_genome().write_fasta(tmp_path / "g.fa")
    good = util.bam_record(name="a", flag=0x63, pos=1000, npos=1200, tlen=350)
    cases = {
        "rg_type": util.bam_record(name="b", flag=0x63, tags=(("RG", "i", 5), ("NM", "C", 0), ("AS", "C", 150))),
        "no_mate_flag": util.bam_record(name="c", flag=0x1, tags=(("RG", "Z", "L1"), ("NM", "C", 0), ("AS", "C", 150))),
        "no_as": util.bam_record(name="d", flag=0x63, tags=(("RG", "Z", "L1"), ("NM", "C", 0))),
    }
    for name, bad in cases.items():
        bam = tmp_path / (name + ".bam")
        bam.write_bytes(util.bam_stream([good, bad]))
        for exe in exes:
            r = subprocess.run([exe, "-r", str(tmp_path / "g.fa"), "-c", "chr1", "-o", str(tmp_path / "x.bamqc"), str(bam)], capture_output=True, text=True)
            assert r.returncode == 1, (name, exe, r.stderr)
