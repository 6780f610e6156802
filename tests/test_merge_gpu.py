"""The multi-GPU plan on one GPU: two engines process the two genome slices of dist.shard_regions(world=2) and are
merged (a) with bqc_merge_from and (b) through the export -> sum -> import path that bamqc_b200.dist drives over
NCCL.  Both must equal the oracle on the whole, coordinate-sorted BAM -- including the coverage histogram, which is
only additive because the slices are separated by re-anchoring gaps."""
import numpy as np
import pytest

import bqc_testutil as util

pytestmark = pytest.mark.gpu


def _split_by_contig(records, offsets, n_contigs):
    """{rid: (lo, hi) record index range}; rid -1 = unmapped tail."""
    rids = np.array([int(np.frombuffer(records[int(o) + 4:int(o) + 8].tobytes(), dtype=np.int32)[0]) for o in offsets[:-1]])
    out = {}
    for rid in list(range(n_contigs)) + [-1]:
        idx = np.nonzero(rids == rid)[0]
        if idx.size:
            assert idx[-1] - idx[0] + 1 == idx.size
            out[rid] = (int(idx[0]), int(idx[-1]) + 1)
    return out


def test_two_shards_merge_exactly(tmp_path):
    import torch
    from bamqc_b200 import Engine, synth, dist
    genome = util.small_genome(seed=21, lengths=(400000, 300000, 100000))
    shards = []
    for rank in range(2):
        lib_ = synth.Library(seed=500 + rank, n_pairs=6000, regions=dist.shard_regions(genome.lengths, rank, 2),
                             first_pair_id=rank * 10 ** 6)
        shards.append((lib_,) + synth.generate(genome, lib_))
    # whole BAM in coordinate order: per contig slice 0 then slice 1, unmapped tails last
    parts = []
    split = [_split_by_contig(rec, offs, 3) for _, rec, offs in shards]
    for rid in [0, 1, 2, -1]:
        for (lib_, rec, offs), sp in zip(shards, split):
            if rid in sp:
                lo, hi = sp[rid]
                parts.append(rec[int(offs[lo]):int(offs[hi])])
    whole = np.concatenate(parts)
    fasta, bam = tmp_path / "g.fa", tmp_path / "whole.ubam"
    genome.write_fasta(fasta)
    synth.write_bam(bam, genome, shards[0][0], whole, whole.size)
    r = util.run_oracle(bam, fasta, tmp_path / "oracle.bamqc", chroms="chr1,chr2")
    assert r.returncode == 0, r.stderr

    def make_engine():
        e = Engine(lane_ids=["L1"], ref_names=genome.names, chroms="chr1,chr2")
        for rid, (p, n) in enumerate(zip(genome.packed, genome.lengths)):
            e.set_reference(rid, p, n)
        return e

    engines = []
    for lib_, rec, offs in shards:
        e = make_engine()
        e.submit(rec, offs)
        e.finish()
        engines.append(e)
    # (b) export -> sum (what the NCCL all-reduce computes) -> import into a fresh engine
    dev = torch.device("cuda", 0)
    c = [torch.empty(e.counters_len(), dtype=torch.int64, device=dev) for e in engines]
    s = [torch.empty(e.sketch_len(), dtype=torch.uint8, device=dev) for e in engines]
    for e, ci, si in zip(engines, c, s):
        e.export_to(ci.data_ptr(), si.data_ptr())
    csum, ssum = c[0] + c[1], s[0] + s[1]
    assert int(ssum.max()) <= 30
    torch.cuda.synchronize()
    third = make_engine()
    third.finish()  # an engine that saw no records still flushes its two empty windows: remove them again
    base = torch.empty(third.counters_len(), dtype=torch.int64, device=dev)
    dummy = torch.empty(third.sketch_len(), dtype=torch.uint8, device=dev)
    third.export_to(base.data_ptr(), dummy.data_ptr())
    third.import_from(csum.data_ptr(), ssum.data_ptr())
    third.write_bamqc("S1", tmp_path / "imported.bamqc")
    # (a) in-process merge
    engines[0].merge_from(engines[1])
    engines[0].write_bamqc("S1", tmp_path / "merged.bamqc")
    for name in ("merged.bamqc", "imported.bamqc"):
        diffs = util.diff_bamqc(tmp_path / "oracle.bamqc", tmp_path / name)
        assert not diffs, name + "\n" + "\n".join(diffs)
    for e in engines + [third]:
        e.close()


def _grown_shards(tmp_path, read_lens):
    """Two engines on GPU 0 whose per-cycle capacities grew along different steps (512 -> 904 for 900 bp reads,
    512 -> 768 for 600 bp reads), the whole BAM in coordinate order and the oracle's .bamqc of it."""
    from bamqc_b200 import Engine, synth, dist
    genome = util.small_genome(seed=22, lengths=(400000, 300000, 100000))
    shards = []
    for rank, L in enumerate(read_lens):
        lib_ = synth.Library(seed=510 + rank, n_pairs=1200, read_len=L, ins_mean=1.6 * L, ins_sd=100, ins_min=L + 50, ins_max=3 * L,
                             regions=dist.shard_regions(genome.lengths, rank, 2), first_pair_id=rank * 10 ** 6)
        shards.append((lib_,) + synth.generate(genome, lib_))
    parts = []
    split = [_split_by_contig(rec, offs, 3) for _, rec, offs in shards]
    for rid in [0, 1, 2, -1]:
        for (lib_, rec, offs), sp in zip(shards, split):
            if rid in sp:
                lo, hi = sp[rid]
                parts.append(rec[int(offs[lo]):int(offs[hi])])
    whole = np.concatenate(parts)
    fasta, bam = tmp_path / "g.fa", tmp_path / "whole.ubam"
    genome.write_fasta(fasta)
    synth.write_bam(bam, genome, shards[0][0], whole, whole.size)
    r = util.run_oracle(bam, fasta, tmp_path / "oracle.bamqc", chroms="chr1,chr2", isize=3000)
    assert r.returncode == 0, r.stderr
    engines = []
    for lib_, rec, offs in shards:
        e = Engine(lane_ids=["L1"], ref_names=genome.names, chroms="chr1,chr2", isize=3000)
        for rid, (p, n) in enumerate(zip(genome.packed, genome.lengths)):
            e.set_reference(rid, p, n)
        e.submit(rec, offs)
        e.finish()
        engines.append(e)
    return genome, engines


def test_merge_engines_that_grew_differently(tmp_path):
    genome, engines = _grown_shards(tmp_path, (900, 600))
    try:
        caps = [e.lib.bqc_read_len_capacity(e.handle) for e in engines]
        assert caps[0] != caps[1] and min(caps) > 512
        engines[0].merge_from(engines[1])
        engines[0].write_bamqc("S1", tmp_path / "merged.bamqc")
        diffs = util.diff_bamqc(tmp_path / "oracle.bamqc", tmp_path / "merged.bamqc")
        assert not diffs, "\n".join(diffs)
    finally:
        for e in engines:
            e.close()


def test_reserve_to_another_engines_capacity_then_export_import(tmp_path):
    """What dist.reduce_engine does: every engine reserves the largest capacity of the group, then the exported blocks
    have one layout and their sum imported into one engine equals the oracle."""
    import torch
    genome, engines = _grown_shards(tmp_path, (600, 900))
    try:
        cap = max(e.lib.bqc_read_len_capacity(e.handle) for e in engines)
        for e in engines:
            e._check(e.lib.bqc_reserve_read_len(e.handle, cap))
            assert e.lib.bqc_read_len_capacity(e.handle) == cap
        assert engines[0].counters_len() == engines[1].counters_len()
        dev = torch.device("cuda", 0)
        c = [torch.empty(e.counters_len(), dtype=torch.int64, device=dev) for e in engines]
        s = [torch.empty(e.sketch_len(), dtype=torch.uint8, device=dev) for e in engines]
        for e, ci, si in zip(engines, c, s):
            e.export_to(ci.data_ptr(), si.data_ptr())
        torch.cuda.synchronize()
        engines[0].import_from((c[0] + c[1]).data_ptr(), (s[0] + s[1]).data_ptr())
        torch.cuda.synchronize()
        engines[0].write_bamqc("S1", tmp_path / "imported.bamqc")
        diffs = util.diff_bamqc(tmp_path / "oracle.bamqc", tmp_path / "imported.bamqc")
        assert not diffs, "\n".join(diffs)
    finally:
        for e in engines:
            e.close()


@pytest.mark.parametrize("devices", ["0,0", "0,1"])
def test_cli_devices_pieces_with_different_longest_reads(tmp_path, devices):
    """bamqualcheck --devices: the first third of the file holds 900 bp reads, the rest only 600 bp reads, so the
    engines of the two pieces grow to different capacities before their tables are merged (~10 MB of BGZF file: the
    command gives every piece at least 4 MB)."""
    import torch
    from bamqc_b200 import synth
    if len(set(devices.split(","))) > torch.cuda.device_count():
        pytest.skip("needs %d GPUs" % len(set(devices.split(","))))
    genome = util.small_genome(seed=24, lengths=(400000, 300000, 100000))
    libs = [synth.Library(seed=520, n_pairs=5000, read_len=900, ins_mean=1500, ins_sd=100, ins_min=950, ins_max=2700,
                          regions={0: (0, 400000)}, emit_unmapped_tail=0),
            synth.Library(seed=521, n_pairs=14000, read_len=600, ins_mean=1000, ins_sd=100, ins_min=650, ins_max=1800,
                          regions={1: (0, 300000)}, first_pair_id=10 ** 6)]
    parts = []
    for lib_ in libs:
        rec, offs = synth.generate(genome, lib_)
        parts.append(rec[:int(offs[-1])])
    whole = np.concatenate(parts + [np.zeros(64, dtype=np.uint8)])
    n = whole.size - 64
    assert parts[0].size < n // 2   # the cut falls among the 600 bp reads
    fasta, ubam, bam = tmp_path / "g.fa", tmp_path / "whole.ubam", tmp_path / "whole.bam"
    genome.write_fasta(fasta)
    synth.write_bam(ubam, genome, libs[0], whole, n)
    synth.write_bam(bam, genome, libs[0], whole, n, level=1)
    r = util.run_oracle(ubam, fasta, tmp_path / "oracle.bamqc", chroms="chr1,chr2")
    assert r.returncode == 0, r.stderr
    g = util.run_cli(["-r", fasta, "-c", "chr1,chr2", "-o", tmp_path / "gpu.bamqc", "--timing", "--devices", devices, bam])
    assert g.returncode == 0, g.stderr + g.stdout
    assert "devices=2" in g.stderr and "could not be cut" not in g.stderr, g.stderr
    diffs = util.diff_bamqc(tmp_path / "oracle.bamqc", tmp_path / "gpu.bamqc")
    assert not diffs, "\n".join(diffs)


@pytest.mark.parametrize("cuts", [(0.37,), (0.0, 0.52), (0.25, 0.25, 0.81)])
def test_one_sorted_stream_cut_at_arbitrary_records(tmp_path, cuts):
    """SURVEY 8e "the exception": ONE gap-free coordinate-sorted BAM cut at arbitrary record indices (also in the middle
    of a pile of reads, with empty pieces) across engines in shard mode.  Everything adds up; the coverage windows are
    resolved with the bqc_cov_shard_* protocol.  The merged result must be byte-identical to the oracle on the whole
    file -- no re-anchoring gaps in the data."""
    from bamqc_b200 import Engine, synth, dist
    genome = util.small_genome(seed=23, lengths=(300000, 200000, 50000))
    lib_ = synth.Library(seed=77, n_pairs=15000)
    records, offsets = synth.generate(genome, lib_)
    n = len(offsets) - 1
    fasta, bam = tmp_path / "g.fa", tmp_path / "whole.ubam"
    genome.write_fasta(fasta)
    synth.write_bam(bam, genome, lib_, records, int(offsets[-1]))
    r = util.run_oracle(bam, fasta, tmp_path / "oracle.bamqc", chroms="chr1,chr2")
    assert r.returncode == 0, r.stderr
    bounds = [0] + [int(n * c) for c in cuts] + [n]
    engines = []
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        e = Engine(lane_ids=["L1"], ref_names=genome.names, chroms="chr1,chr2", staging_bytes=8 << 20)
        for rid, (p, m) in enumerate(zip(genome.packed, genome.lengths)):
            e.set_reference(rid, p, m)
        e.cov_defer(2 if (lo == 0 and len(cuts) != 2) else 1)   # the first piece may run like a stand-alone engine
        # several submissions per piece: the records that take part are collected across batches
        step = max(1, (hi - lo) // 3)
        for a in range(lo, hi, step):
            b = min(hi, a + step)
            o = offsets[a:b + 1]
            e.submit(records[int(o[0]):int(o[-1])], None)
        e.finish()
        engines.append(e)
    delta = dist.resolve_coverage_local(engines)
    for e in engines[1:]:
        engines[0].merge_from(e)
    engines[0].poscov_adjust(delta)
    engines[0].write_bamqc("S1", tmp_path / "merged.bamqc")
    diffs = util.diff_bamqc(tmp_path / "oracle.bamqc", tmp_path / "merged.bamqc")
    for e in engines:
        e.close()
    assert not diffs, "\n".join(diffs)
