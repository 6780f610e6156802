"""The kernel variants the engine selects from -e, -k, -q, the read groups and the BQC_* switches, the k_stats epochs
and the shared-memory bins that spill to global memory, each against the CPU oracle: the `.bamqc` text byte for byte
and, wherever a sketch exists, the raw sketch, the F2 table and sumCount of every (lane, q, k).  Every variant test
also checks which kernels ran, so that a dispatch that falls back to the default kernel fails."""
import numpy as np
import pytest

import bqc_testutil as util

pytestmark = pytest.mark.gpu

V2_640 = "k_sketch32v2<640u>"
K32 = "bqc::k_sketch32("        # k_sketch32 (not k_sketch32v2)
GEN_SMEM = "k_sketch<true>"     # generic k_sketch, F2 table in shared memory
GEN_GLOBAL = "k_sketch<false>"  # generic k_sketch, F2 table in global memory


def _short_reads(klist, lanes, seed):
    """Unmapped pairs (appended after the unmapped tail, so coordinate order holds) of lengths k-1, k and k+1 for every
    k, with N bases at the edges of the first and last window, at qualities around the cutoffs."""
    rng = np.random.default_rng(seed)
    recs = []
    for k in klist:
        for L in (k - 1, k, k + 1):
            if L < 1:
                continue
            for n_at in (None, 0, k - 1, L - 1, L - k):
                for q in (40, 94, 200, 222):
                    seq = list("ACGT"[c] for c in rng.integers(0, 4, L))
                    if n_at is not None and 0 <= n_at < L:
                        seq[n_at] = "N"
                    for lane in lanes:
                        for flag in (0x4D, 0x9D):  # unmapped pair, first / second mate, reverse or not
                            recs.append(util.bam_record(name=f"s{len(recs)}", flag=flag, rid=-1, pos=-1, mapq=0, cigar=(), seq="".join(seq),
                                                        qual=[q] * L, nrid=-1, npos=-1, tlen=0, tags=(("RG", "Z", lane),)))
    return b"".join(recs)


def _parity(tmp_path, lib_, klist=(32,), qlist=(17,), e=0.01, isize=1000, seed=1, mutate=True, extra_short=True,
            mode="offsets", engine_kwargs=None):
    """Synthetic library (+ QUAL mutator, + short reads) through the oracle and the engine; returns the kernel names."""
    from bamqc_b200 import synth
    genome = util.small_genome()
    records, offsets = synth.generate(genome, lib_)
    n = int(offsets[-1])
    if mutate:
        util.mutate_qual(records, offsets, share=0.5, seed=lib_.seed)
    if extra_short:
        extra = np.frombuffer(_short_reads(klist, synth.lane_ids(lib_), lib_.seed), dtype=np.uint8)
        p, ends = 0, []
        while p < extra.size:
            p += 4 + int(extra[p:p + 4].view(np.int32)[0])
            ends.append(p)
        records = np.concatenate([records[:n], extra, np.zeros(64, dtype=np.uint8)])
        offsets = np.concatenate([offsets, n + np.array(ends, dtype=np.uint64)])
        n = int(offsets[-1])
    tmp_path.mkdir(exist_ok=True)
    fasta, bam = tmp_path / "ref.fa", tmp_path / "in.ubam"
    genome.write_fasta(fasta)
    synth.write_bam(bam, genome, lib_, records, n)
    r = util.run_oracle(bam, fasta, tmp_path / "oracle.bamqc", chroms="chr1,chr2", isize=isize, klist=klist, qlist=qlist,
                        e=e, seed=seed, dump=tmp_path / "oracle.dump")
    assert r.returncode == 0, r.stderr
    eng, names = util.kernel_names(lambda: util.run_engine(
        genome, lib_, records, offsets, tmp_path / "gpu.bamqc", chroms="chr1,chr2", isize=isize, klist=klist, qlist=qlist,
        e=e, seed=seed, keep=True, mode=mode, engine_kwargs=engine_kwargs))
    try:
        assert eng.records_seen == len(offsets) - 1
        diffs = util.diff_bamqc(tmp_path / "oracle.bamqc", tmp_path / "gpu.bamqc")
        assert not diffs, "\n".join(diffs)
        util.assert_sketches_equal(eng, tmp_path / "oracle.dump", synth.lane_ids(lib_), len(qlist) * len(klist))
    finally:
        eng.close()
    return names


# ---- A. sketch geometry (-e), k, q cutoff and the sketch kernels ------------------------------------------------------
# -e -> (sketch words per level / 2, F2 table): 0.2 -> 512 / 64 (numcounts clamp), 0.05 -> 2048 / 1024,
# 0.008 -> 65536 / 32768 (the v2 kernel with sk_size != f2size), 0.005 -> 131072 / 131072 (F2 table in global memory).
# q cutoffs: (char)(33 + q) is 33..127 up to q = 94 (k_sketch32v2); from 95 on it is negative (k_sketch32).
@pytest.mark.parametrize("e,klist,qlist,ran,not_ran", [
    (0.2, (1, 32), (0, 17, 94), (V2_640, GEN_SMEM), (K32, GEN_GLOBAL)),
    (0.05, (15, 32, 33), (95, 200), (K32, GEN_SMEM), ("k_sketch32v2", GEN_GLOBAL)),
    (0.008, (31, 32), (17, 100), (V2_640, K32, GEN_SMEM), (GEN_GLOBAL,)),
    (0.005, (32, 63), (17, 200), (GEN_GLOBAL,), ("k_sketch32", GEN_SMEM)),
], ids=["e0.2", "e0.05", "e0.008", "e0.005"])
def test_sketch_geometry_and_kernels(tmp_path, e, klist, qlist, ran, not_ran):
    from bamqc_b200 import synth
    names = _parity(tmp_path, synth.Library(seed=601, n_pairs=2500), klist=klist, qlist=qlist, e=e)
    util.assert_kernels(names, ran, not_ran)


@pytest.mark.parametrize("v2,kernel", [(0, K32), (1, "k_sketch32v2<1024u>"), (2, "k_sketch32v2<512u>"), (4, "k_sketch32v2<768u>")])
def test_sketch_v2_switch(tmp_path, monkeypatch, v2, kernel):
    from bamqc_b200 import synth
    monkeypatch.setenv("BQC_SKETCH_V2", str(v2))
    names = _parity(tmp_path, synth.Library(seed=610 + v2, n_pairs=2500), qlist=(0, 17, 94))
    util.assert_kernels(names, (kernel,), (V2_640,) + (("k_sketch32v2",) if v2 == 0 else ()))


@pytest.mark.parametrize("threads", [256, 1024])
def test_sketch32_threads(tmp_path, monkeypatch, threads):
    from bamqc_b200 import synth
    monkeypatch.setenv("BQC_SKETCH_THREADS", str(threads))
    names = _parity(tmp_path, synth.Library(seed=620, n_pairs=2500), qlist=(95, 17))
    util.assert_kernels(names, (K32, V2_640))


def test_two_lanes_several_qk(tmp_path):
    """Per-(lane, q/k) sketch offsets differ for every pair."""
    from bamqc_b200 import synth
    names = _parity(tmp_path, synth.Library(seed=630, n_pairs=3000, n_lanes=2), klist=(15, 32), qlist=(17, 94, 95))
    util.assert_kernels(names, (V2_640, K32, GEN_SMEM), (GEN_GLOBAL,))


# ---- B. table-kernel switches: stress library at -q 2,17 (populated sketches) and 2 x 251 bp reads ----------------------
SWITCHES = {
    "tickets0": ({"BQC_TICKETS": "0"}, ("k_stats<1>",), ()),
    "tickets2": ({"BQC_TICKETS": "2"}, ("k_stats<1>",), ()),
    "stage2": ({"BQC_STATS_STAGE": "2"}, ("k_stats<2>",), ("k_stats<1>",)),
    "cov_overlap0": ({"BQC_COV_OVERLAP": "0"}, ("k_cov_tiles", "k_stats<1>"), ()),
    "cov_overlap1": ({"BQC_COV_OVERLAP": "1"}, ("k_cov_tiles", "k_stats<1>"), ()),
    "cov_bps1": ({"BQC_COV_BPS": "1"}, ("k_cov_tiles",), ()),
    "stats_bps1": ({"BQC_STATS_BPS": "1"}, ("k_stats<1>",), ()),
}


@pytest.mark.parametrize("name", sorted(SWITCHES))
def test_table_kernel_switch(tmp_path, monkeypatch, name):
    from bamqc_b200 import synth
    env, ran, not_ran = SWITCHES[name]
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    names = _parity(tmp_path / "stress", synth.Library(seed=640, n_pairs=6000).stress(), qlist=(2, 17), mutate=False, extra_short=False)
    util.assert_kernels(names, ran, not_ran)
    names = _parity(tmp_path / "long", synth.Library(seed=641, n_pairs=1500, read_len=251, ins_mean=450), qlist=(2, 17), mutate=True,
                    extra_short=False, mode="whole")
    util.assert_kernels(names, ran, not_ran)


def test_lane_index_switch_three_lanes(tmp_path, monkeypatch):
    """BQC_LANE_INDEX=0: the staged k_stats filters the lanes over the whole batch instead of the lane-indexed k_stats<0>."""
    from bamqc_b200 import synth
    monkeypatch.setenv("BQC_LANE_INDEX", "0")
    names = _parity(tmp_path, synth.Library(seed=650, n_pairs=4000, n_lanes=3).stress(), qlist=(2, 17), mutate=False, extra_short=False)
    util.assert_kernels(names, ("k_stats<1>",), ("k_stats<0>",))


def test_inflate_streams_switch(tmp_path, monkeypatch):
    """BQC_INFLATE_STREAMS=1: every k_inflate on the framing stream."""
    from bamqc_b200 import Engine, synth
    monkeypatch.setenv("BQC_INFLATE_STREAMS", "1")
    genome = util.small_genome()
    lib_ = synth.Library(seed=660, n_pairs=8000).stress()
    records, offsets = synth.generate(genome, lib_)
    n = int(offsets[-1])
    fasta, bam = tmp_path / "ref.fa", tmp_path / "in.ubam"
    genome.write_fasta(fasta)
    synth.write_bam(bam, genome, lib_, records, n)
    r = util.run_oracle(bam, fasta, tmp_path / "oracle.bamqc", chroms="chr1,chr2", qlist=(2, 17), dump=tmp_path / "oracle.dump")
    assert r.returncode == 0, r.stderr
    comp = synth.bgzf_compress(records[:n], level=6)
    starts = util.bgzf_block_starts(comp)
    cuts = [0, starts[len(starts) // 3], starts[2 * len(starts) // 3], comp.size]

    def run():
        eng = Engine(lane_ids=["L1"], ref_names=genome.names, chroms="chr1,chr2", qlist=(2, 17), staging_bytes=1 << 20)
        for rid, (p, m) in enumerate(zip(genome.packed, genome.lengths)):
            eng.set_reference(rid, p, m)
        for i in range(3):
            eng.submit_bgzf(comp[cuts[i]:cuts[i + 1]], last=i == 2)
        eng.finish()
        return eng

    eng, names = util.kernel_names(run)
    try:
        assert eng.records_seen == len(offsets) - 1
        eng.write_bamqc("S1", tmp_path / "gpu.bamqc")
        diffs = util.diff_bamqc(tmp_path / "oracle.bamqc", tmp_path / "gpu.bamqc")
        assert not diffs, "\n".join(diffs)
        util.assert_sketches_equal(eng, tmp_path / "oracle.dump", ["L1"], 2)
    finally:
        eng.close()
    util.assert_kernels(names, ("k_inflate", "k_frame_emit"))


# ---- C. k_stats epochs at their bounds ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def epoch_data(tmp_path_factory):
    """One lane, 50 bp reads, every read first-in-pair, forward and with the same sequence, quality 222 on 7 of 8 reads:
    one (mate, base, cycle) cell takes all 256 records of a CTA iteration, 3584 of its 4095 counts and ~796 k of its 2^20
    quality per epoch.  3 epochs for every CTA of one CTA per SM."""
    import torch
    d = tmp_path_factory.mktemp("epochs")
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    n = 3 * 14 * 256 * n_sm + 1001
    genome = util.small_genome()
    seq = "ACGTTGCAAC" * 5
    rec = [np.frombuffer(util.bam_record(name="e", flag=0x63, rid=0, pos=0, cigar=((50, "M"),), seq=seq, qual=[q] * 50, npos=0, tlen=350,
                                         tags=(("RG", "Z", "L1"), ("NM", "C", 0), ("AS", "C", 50))), dtype=np.uint8) for q in (222, 30)]
    arr = np.tile(rec[0], (n, 1))
    arr[7::8] = rec[1]
    pos = (1000 + np.arange(n) // 8).astype(np.int32)
    arr[:, 8:12] = pos.view(np.uint8).reshape(n, 4)
    arr[:, 28:32] = (pos + 300).view(np.uint8).reshape(n, 4)
    records = arr.reshape(-1)
    refs = list(zip(genome.names, genome.lengths))
    bam = d / "in.ubam"
    with open(bam, "wb") as f:
        f.write(util.bam_stream([], refs=refs))
        f.write(records.tobytes())
    fasta = d / "ref.fa"
    genome.write_fasta(fasta)
    r = util.run_oracle(bam, fasta, d / "oracle.bamqc", chroms="chr1,chr2", dump=d / "oracle.dump")
    assert r.returncode == 0, r.stderr
    return d, genome, records, n


@pytest.mark.parametrize("tickets", ["1", "0"])
def test_stats_epochs_full_cells(epoch_data, tmp_path, monkeypatch, capfd, tickets):
    from bamqc_b200 import Engine
    d, genome, records, n = epoch_data
    monkeypatch.setenv("BQC_STATS_BPS", "1")
    monkeypatch.setenv("BQC_TICKETS", tickets)
    monkeypatch.setenv("BQC_TRACE", "1")
    eng = Engine(lane_ids=["L1"], ref_names=genome.names, chroms="chr1,chr2")
    try:
        for rid, (p, m) in enumerate(zip(genome.packed, genome.lengths)):
            eng.set_reference(rid, p, m)
        eng.submit(np.concatenate([records, np.zeros(64, dtype=np.uint8)]), None, n_bytes=records.size)
        eng.finish()
        assert eng.records_seen == n
        eng.write_bamqc("S1", tmp_path / "gpu.bamqc")
        err = capfd.readouterr().err
        assert f"n={n}\n" in err, err[-2000:]   # one batch
        diffs = util.diff_bamqc(d / "oracle.bamqc", tmp_path / "gpu.bamqc")
        assert not diffs, "\n".join(diffs)
        util.assert_sketches_equal(eng, d / "oracle.dump", ["L1"], 1)
    finally:
        eng.close()


# ---- D. shared-memory bins that spill to global memory (through the drop-in command) ---------------------------------
def test_spill_bins(tmp_path):
    recs = []
    pos = 1000

    def add(first=None, **kw):
        nonlocal pos
        pos += 13
        i = len(recs)
        first = i % 2 == 0 if first is None else first
        kw.setdefault("tags", (("RG", "Z", "L1"), ("NM", "C", 0), ("AS", "C", 150)))
        kw.setdefault("tlen", 350 if first else -350)
        recs.append(util.bam_record(name=f"p{i}", flag=0x63 if first else 0x93, rid=0, pos=pos, npos=pos + 200, **kw))

    # average / ceil quality >= 64 (up to 222)
    for q in (63, 64, 65, 100, 150, 199, 200, 221, 222):
        add(qual=[q] * 150)
    add(qual=[64 + (j % 159) for j in range(150)])
    add(qual=[222] * 149 + [221])
    # NM - D - I around the 32 shared-memory bins
    for x in (31, 32, 33, 120):
        add(cigar=((60, "M"), (3, "D"), (2, "I"), (88, "M")), tags=(("RG", "Z", "L1"), ("NM", "i", x + 5), ("AS", "C", 140)))
    # summed insertions around 32
    for ins in ((31,), (32,), (20, 20), (33,)):
        cig = [(40, "M")]
        for k in ins:
            cig += [(k, "I"), (10, "M")]
        cig[-1] = (150 - 40 - sum(ins) - 10 * (len(ins) - 1), "M")
        add(cigar=tuple(cig), tags=(("RG", "Z", "L1"), ("NM", "i", sum(ins)), ("AS", "C", 100)))
    add(mapq=255)
    add(mapq=254)
    # insert sizes around the 4096 shared-memory bins and the -i 10000 capacity
    for t in (0, 4087, 4088, 4095, 4096, 4097, 9999, 10000, 10001, 2147483647):
        for sgn in (1, -1):
            add(tlen=sgn * t, first=True)
            add(tlen=-sgn * t, first=False)
    util.against_oracle(tmp_path, util.bam_stream(recs), opts=("-c", "chr1,chr2", "-i", "10000"))
