"""Parity at the stated size of BASELINE.json's correctness configuration (cfg 1: 1 M synthetic 2x150 bp records on a
10 Mb chr1, seed 20260101, defaults) and of the stress library at the same size (cfg 4): the CUDA path through the C
ABI and through the drop-in command must give a `.bamqc` that is byte-identical to the CPU oracle AND to
oracle/_ref/bamqualcheck_ref (the reference's own statistics code), plus identical raw sketch and F2 tables.  Sizes
matter: 32-bit shared-memory counters, 16-bit 8-mer fields, the per-warp k-mer counters and the coverage tiling all
depend on them."""
import os
import subprocess
import warnings

import numpy as np
import pytest

import bqc_testutil as util

pytestmark = pytest.mark.gpu


def _full_size(tmp_path, stress):
    from bamqc_b200 import synth
    genome = synth.Genome.make(20260101, ["chr1"], [10_000_000])
    lib_ = synth.Library(seed=20260104 if stress else 20260101, n_pairs=497_500)
    if stress:
        lib_.stress()
    records, offsets = synth.generate(genome, lib_)
    n = len(offsets) - 1
    assert 990_000 <= n <= 1_010_000
    fasta, bam = tmp_path / "ref.fa", tmp_path / "in.ubam"
    genome.write_fasta(fasta)
    synth.write_bam(bam, genome, lib_, records, int(offsets[-1]))
    r = util.run_oracle(bam, fasta, tmp_path / "oracle.bamqc", dump=tmp_path / "oracle.dump")
    assert r.returncode == 0, r.stderr
    # (1) the C ABI, three submissions cut anywhere in the byte stream (device framing)
    eng = util.run_engine(genome, lib_, records, offsets, tmp_path / "gpu.bamqc", chroms=",".join("chr%d" % i for i in range(1, 23)),
                          keep=True, mode="stream", chunk_bytes=int(offsets[-1]) // 3 + 7)
    try:
        assert eng.records_seen == n
        diffs = util.diff_bamqc(tmp_path / "oracle.bamqc", tmp_path / "gpu.bamqc")
        assert not diffs, "\n".join(diffs)
        table, f2 = util.oracle_sketch(tmp_path / "oracle.dump", 1)[0]
        assert np.array_equal(eng.sketch(0, 0), table)
        assert np.array_equal(eng.table("F2TABLE", 0, 0), f2)
    finally:
        eng.close()
    # (2) the drop-in command on the same files vs the reference's own code
    r = util.run_cli(["-r", fasta, "-o", tmp_path / "cli.bamqc", bam])
    assert r.returncode == 0, r.stderr
    assert open(tmp_path / "cli.bamqc", "rb").read() == open(tmp_path / "oracle.bamqc", "rb").read()
    if os.path.exists(util.REF_BIN):
        r = subprocess.run([util.REF_BIN, "-r", str(fasta), "-o", str(tmp_path / "ref.bamqc"), str(bam)], capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert open(tmp_path / "cli.bamqc", "rb").read() == open(tmp_path / "ref.bamqc", "rb").read()
    else:
        warnings.warn("oracle/_ref not built: the 1 M-record .bamqc was compared with the oracle only, not with the reference build")


def test_cfg1_one_million_records(tmp_path):
    _full_size(tmp_path, stress=False)


def test_cfg4_stress_library_one_million_records(tmp_path):
    _full_size(tmp_path, stress=True)
