"""Parity of the CUDA path (through the C ABI) against the CPU oracle on seeded synthetic data.
Bit-exact for every integer table; the `.bamqc` text (which also carries the derived doubles at the
reference's 6 significant digits) must be byte-identical."""
import numpy as np
import pytest

import bqc_testutil as util

pytestmark = pytest.mark.gpu


def _roundtrip(tmp_path, lib_, genome=None, chroms="chr1,chr2", isize=1000, klist=(32,), qlist=(17,), seed=1,
               n_batches=1, resident=False, engine_kwargs=None, mode="offsets", chunk_bytes=None, expect_repaired=None):
    from bamqc_b200 import synth
    genome = genome or util.small_genome()
    records, offsets = synth.generate(genome, lib_)
    n_bytes = int(offsets[-1])
    fasta, bam = tmp_path / "ref.fa", tmp_path / "in.ubam"
    genome.write_fasta(fasta)
    synth.write_bam(bam, genome, lib_, records, n_bytes)
    r = util.run_oracle(bam, fasta, tmp_path / "oracle.bamqc", chroms=chroms, isize=isize, klist=klist, qlist=qlist,
                        seed=seed, dump=tmp_path / "oracle.dump")
    assert r.returncode == 0, r.stderr
    eng = util.run_engine(genome, lib_, records, offsets, tmp_path / "gpu.bamqc", chroms=chroms, isize=isize,
                          klist=klist, qlist=qlist, seed=seed, n_batches=n_batches, resident=resident,
                          engine_kwargs=engine_kwargs, keep=True, mode=mode, chunk_bytes=chunk_bytes)
    try:
        assert eng.records_seen == len(offsets) - 1
        if expect_repaired is not None:
            assert (eng.frames_repaired > 0) == expect_repaired
        diffs = util.diff_bamqc(tmp_path / "oracle.bamqc", tmp_path / "gpu.bamqc")
        assert not diffs, "\n".join(diffs)
        # sketch tables and F2 tables themselves, not only the estimators printed in the text
        util.assert_sketches_equal(eng, tmp_path / "oracle.dump", synth.lane_ids(lib_), len(qlist) * len(klist))
    finally:
        eng.close()


def test_standard_library(tmp_path):
    from bamqc_b200 import synth
    _roundtrip(tmp_path, synth.Library(seed=11, n_pairs=20000))


# The stress library's qualities leave no window of 32 bases at the default cutoff 17: its roundtrips add -q 2 so that
# they compare populated sketches too.
def test_stress_library(tmp_path):
    from bamqc_b200 import synth
    _roundtrip(tmp_path, synth.Library(seed=12, n_pairs=15000).stress(), qlist=(2, 17))


def test_many_batches_and_long_insert(tmp_path):
    from bamqc_b200 import synth
    lib_ = synth.Library(seed=13, n_pairs=12000, ins_mean=1500, ins_sd=400, ins_min=150, ins_max=6000)
    _roundtrip(tmp_path, lib_, isize=3000, n_batches=7)


def test_resident_replay(tmp_path):
    from bamqc_b200 import synth
    _roundtrip(tmp_path, synth.Library(seed=14, n_pairs=9000), n_batches=3, resident=True)


def test_two_lanes_and_kq_grid(tmp_path):
    from bamqc_b200 import synth
    _roundtrip(tmp_path, synth.Library(seed=15, n_pairs=8000, n_lanes=2), klist=(15, 32, 63), qlist=(10, 17))


def test_sparse_coverage_windows(tmp_path):
    """Mean gap between reads ~ 600 bp: exercises window rolls, resets and the tiny-ring segmentation."""
    from bamqc_b200 import synth
    genome = util.small_genome(seed=9, lengths=(3000000, 2000000, 500000))
    lib_ = synth.Library(seed=16, n_pairs=4000)
    _roundtrip(tmp_path, lib_, genome=genome, n_batches=2, engine_kwargs=dict(cov_ring_log2=13))


def test_other_read_length_and_seed(tmp_path):
    from bamqc_b200 import synth
    _roundtrip(tmp_path, synth.Library(seed=17, n_pairs=6000, read_len=101, ins_mean=300), seed=5)


# ---- device-side framing (kernel_frame.cuh): the engine finds the record boundaries itself ----------------------
def test_stats_direct_path_switch(tmp_path, monkeypatch):
    """BQC_STATS_STAGE=0: k_stats reads the records straight from global memory instead of through the per-warp
    shared-memory staging (same statements, other loaders); stress library so that clipped / indel reads are common."""
    from bamqc_b200 import synth
    monkeypatch.setenv("BQC_STATS_STAGE", "0")
    lib_ = synth.Library(seed=31, n_pairs=6000)
    lib_.stress()
    _roundtrip(tmp_path, lib_, qlist=(2, 17))


def test_long_reads_split_the_staging_span(tmp_path):
    """2 x 250 bp: the 32 records of a warp (~15 KB) do not fit the 10 KB staging area of k_stats and are staged in
    pieces; also an odd read length for the reverse-read nibble windows."""
    from bamqc_b200 import synth
    _roundtrip(tmp_path, synth.Library(seed=32, n_pairs=4000, read_len=251, ins_mean=450))


def test_tables_grow_with_the_longest_read(tmp_path):
    """2 x 700 bp with the default per-cycle capacity of 512: the result block is moved to a larger layout when the first
    batch with longer reads arrives (the reference's String<>s grow the same way, src/QualityCheck.hpp:85-109); the
    second half of the records comes in a later batch."""
    from bamqc_b200 import synth
    _roundtrip(tmp_path, synth.Library(seed=33, n_pairs=1500, read_len=700, ins_mean=1200, ins_sd=100, ins_min=800, ins_max=2000), n_batches=2)


def test_very_long_reads_without_staging(tmp_path):
    """2 x 1500 bp: the per-cycle rows leave no room for the per-warp staging areas; k_stats reads the records from global memory."""
    from bamqc_b200 import synth
    _roundtrip(tmp_path, synth.Library(seed=34, n_pairs=400, read_len=1500, ins_mean=2500, ins_sd=100, ins_min=1800, ins_max=4000), isize=3000)


def test_device_framing_whole_record_slices(tmp_path):
    from bamqc_b200 import synth
    _roundtrip(tmp_path, synth.Library(seed=21, n_pairs=20000), n_batches=3, mode="whole", expect_repaired=False)


def test_stream_chunks_cut_records_anywhere(tmp_path):
    """Chunks of 1,000,003 bytes: every chunk ends inside a record; the partial record is carried on the device."""
    from bamqc_b200 import synth
    _roundtrip(tmp_path, synth.Library(seed=22, n_pairs=20000).stress(), qlist=(2, 17), mode="stream", chunk_bytes=1000003,
               expect_repaired=False)


def test_stream_tiny_chunks_and_tiny_staging(tmp_path):
    """Chunks smaller than a record and than the speculation window; staging buffers of 64 KiB."""
    from bamqc_b200 import synth
    _roundtrip(tmp_path, synth.Library(seed=23, n_pairs=1500), mode="stream", chunk_bytes=173,
               engine_kwargs=dict(staging_bytes=1 << 16), expect_repaired=False)
    _roundtrip(tmp_path, synth.Library(seed=24, n_pairs=6000), mode="stream", chunk_bytes=50021,
               engine_kwargs=dict(staging_bytes=1 << 16), expect_repaired=False)


def test_stream_repair_path(tmp_path, monkeypatch):
    """Every speculation is declared failed: k_frame_repair frames sequentially, results are the same."""
    from bamqc_b200 import synth
    monkeypatch.setenv("BQC_FRAME_FORCE_REPAIR", "1")
    _roundtrip(tmp_path, synth.Library(seed=25, n_pairs=5000), mode="stream", chunk_bytes=300007, expect_repaired=True)


def test_stream_host_framing_switch(tmp_path, monkeypatch):
    """BQC_HOST_FRAMING=1: same stream API, records framed by the host framer."""
    from bamqc_b200 import synth
    monkeypatch.setenv("BQC_HOST_FRAMING", "1")
    _roundtrip(tmp_path, synth.Library(seed=26, n_pairs=5000), mode="stream", chunk_bytes=300007, expect_repaired=False)


def test_stream_two_lanes_on_the_device_framer(tmp_path):
    """Several read groups: the lane of every record comes from its RG tag on the device (k_frame_lanes), so the
    stream keeps device-side framing."""
    from bamqc_b200 import synth
    _roundtrip(tmp_path, synth.Library(seed=27, n_pairs=5000, n_lanes=2), mode="stream", chunk_bytes=400009, expect_repaired=False)


def test_stream_three_lanes_with_host_framing_switch(tmp_path, monkeypatch):
    """BQC_HOST_FRAMING=1: the host framer and the host RG lookup (same results)."""
    from bamqc_b200 import synth
    monkeypatch.setenv("BQC_HOST_FRAMING", "1")
    _roundtrip(tmp_path, synth.Library(seed=29, n_pairs=4000, n_lanes=3), mode="stream", chunk_bytes=500009)


def test_stream_truncated_record_is_an_error(tmp_path):
    from bamqc_b200 import Engine, synth
    from bamqc_b200.engine import BamQCError
    genome = util.small_genome()
    lib_ = synth.Library(seed=28, n_pairs=2000)
    records, offsets = synth.generate(genome, lib_)
    eng = Engine(lane_ids=synth.lane_ids(lib_), ref_names=genome.names, chroms="chr1,chr2")
    try:
        cut = int(offsets[-1]) - 17
        with pytest.raises(BamQCError) as ei:
            eng.submit_stream(records[:cut], last=True)
            eng.finish()
        assert ei.value.code == 4
    finally:
        eng.close()


# ---- device-side BGZF inflate (kernel_inflate.cuh) --------------------------------------------------------------
def _bgzf_roundtrip(tmp_path, lib_, level, pieces=1, with_header=False, engine_kwargs=None, monkey_env=None, mutate=None):
    """Records -> BGZF (zlib at `level`) -> bqc_submit_bgzf -> .bamqc identical to the oracle's."""
    from bamqc_b200 import Engine, synth
    genome = util.small_genome()
    records, offsets = synth.generate(genome, lib_)
    n_bytes = int(offsets[-1])
    if mutate:
        mutate(records, offsets)
    fasta, bam = tmp_path / "ref.fa", tmp_path / "in.ubam"
    genome.write_fasta(fasta)
    synth.write_bam(bam, genome, lib_, records, n_bytes)
    r = util.run_oracle(bam, fasta, tmp_path / "oracle.bamqc", chroms="chr1,chr2")
    assert r.returncode == 0, r.stderr
    payload = records[:n_bytes]
    skip = 0
    if with_header:  # the inflated stream starts with a BAM header that is not block aligned
        raw = np.fromfile(bam, dtype=np.uint8)
        skip = raw.size - n_bytes
        payload = raw
    comp = synth.bgzf_compress(payload, level=level)
    eng = Engine(lane_ids=synth.lane_ids(lib_), ref_names=genome.names, chroms="chr1,chr2", **(engine_kwargs or {}))
    try:
        for rid, (p, n) in enumerate(zip(genome.packed, genome.lengths)):
            eng.set_reference(rid, p, n)
        # cut the compressed bytes at BGZF block boundaries into `pieces` submissions
        starts = util.bgzf_block_starts(comp)
        cuts = [starts[len(starts) * i // pieces] for i in range(pieces)] + [comp.size]
        for i in range(pieces):
            eng.submit_bgzf(comp[cuts[i]:cuts[i + 1]], skip=skip if i == 0 else 0, last=i == pieces - 1)
        eng.finish()
        assert eng.records_seen == len(offsets) - 1
        eng.write_bamqc("S1", tmp_path / "gpu.bamqc")
        diffs = util.diff_bamqc(tmp_path / "oracle.bamqc", tmp_path / "gpu.bamqc")
        assert not diffs, "\n".join(diffs)
    finally:
        eng.close()


@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_device_inflate_levels(tmp_path, level):
    """Stored blocks (level 0), fast and best dynamic-Huffman streams."""
    from bamqc_b200 import synth
    _bgzf_roundtrip(tmp_path, synth.Library(seed=31 + level, n_pairs=6000), level)


def test_device_inflate_header_skip_and_pieces(tmp_path):
    from bamqc_b200 import synth
    _bgzf_roundtrip(tmp_path, synth.Library(seed=41, n_pairs=9000).stress(), 6, pieces=5, with_header=True)


def test_device_inflate_small_staging_splits_submission(tmp_path):
    from bamqc_b200 import synth
    _bgzf_roundtrip(tmp_path, synth.Library(seed=42, n_pairs=5000), 6, engine_kwargs=dict(staging_bytes=1 << 18))


def test_device_inflate_tiny_input_fixed_huffman(tmp_path):
    """A few records: zlib emits fixed-Huffman blocks for tiny inputs."""
    from bamqc_b200 import synth
    _bgzf_roundtrip(tmp_path, synth.Library(seed=43, n_pairs=3), 6)
    _bgzf_roundtrip(tmp_path, synth.Library(seed=44, n_pairs=40), 9)


def _repetitive_fields(records, offsets):
    """Overwrite SEQ / QUAL of most records with periodic patterns: zlib then emits long matches (up to 258) at short
    distances -- period 1 (runs), 2..31 (a step of 32 lanes wraps several times), 32..63 (overlapping but longer than a
    warp step) -- next to the ordinary literal-heavy records."""
    periods = [1, 2, 3, 5, 7, 16, 31, 32, 33, 40, 63]
    for i in range(len(offsets) - 1):
        mode = i % 13
        if mode >= len(periods):
            continue
        o = int(offsets[i]) + 4   # past block_size
        l_name = int(records[o + 8])
        n_cig = int(records[o + 12]) | int(records[o + 13]) << 8
        l_seq = int(records[o + 16]) | int(records[o + 17]) << 8 | int(records[o + 18]) << 16
        seq = o + 32 + l_name + 4 * n_cig
        qual = seq + (l_seq + 1) // 2
        per = periods[mode]
        pat_q = (np.arange(per, dtype=np.uint8) * 3 + 5 + mode) % 41
        records[qual:qual + l_seq] = np.resize(pat_q, l_seq)
        if i % 2:   # one-hot nibbles only (A, C, G, T), so the sequence stays a plain read
            pat_s = np.array([0x11, 0x12, 0x48, 0x84, 0x21, 0x88, 0x14], dtype=np.uint8)[(np.arange(per) * 5 + mode) % 7]
            n = l_seq // 2
            records[seq:seq + n] = np.resize(pat_s, n)


@pytest.mark.parametrize("level", [1, 6, 9])
def test_device_inflate_long_overlapping_matches(tmp_path, level):
    from bamqc_b200 import synth
    _bgzf_roundtrip(tmp_path, synth.Library(seed=47 + level, n_pairs=2500, read_len=400, ins_mean=600.0, ins_min=400, ins_max=1000), level,
                    mutate=_repetitive_fields)


def test_device_inflate_corrupt_block_is_an_error(tmp_path):
    from bamqc_b200 import Engine, synth
    from bamqc_b200.engine import BamQCError
    genome = util.small_genome()
    lib_ = synth.Library(seed=45, n_pairs=3000)
    records, offsets = synth.generate(genome, lib_)
    comp = synth.bgzf_compress(records[:int(offsets[-1])], level=6).copy()
    starts = util.bgzf_block_starts(comp)
    comp[starts[2] + 40:starts[2] + 60] ^= 0x5A  # damage the deflate payload of the third block
    eng = Engine(lane_ids=synth.lane_ids(lib_), ref_names=genome.names, chroms="chr1,chr2")
    try:
        with pytest.raises(BamQCError) as ei:
            eng.submit_bgzf(comp, last=True)
            eng.finish()
        assert ei.value.code == 4
    finally:
        eng.close()


def test_bgzf_host_inflate_switch(tmp_path, monkeypatch):
    from bamqc_b200 import synth
    monkeypatch.setenv("BQC_HOST_FRAMING", "1")
    _bgzf_roundtrip(tmp_path, synth.Library(seed=46, n_pairs=4000), 6, pieces=3, with_header=True)
