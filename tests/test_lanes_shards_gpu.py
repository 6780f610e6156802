"""Several read groups (lanes) cut across engines.  Every lane's records, in file order, are a stream of their own for
the coverage windows; cutting the file at record k cuts every lane's stream there, and the shard protocol runs once per
lane (bqc_cov_shard_*_lane, dist.resolve_coverage_shards_lanes).  The oracle's .bamqc of the whole file is the checker,
byte for byte."""
import os

import numpy as np
import pytest

import bqc_testutil as util

pytestmark = pytest.mark.gpu

CUTS = [(0.37,), (0.0, 0.52), (0.25, 0.25, 0.81)]


def _concat(genome, libs):
    """Coordinate-sorted records of several libraries that cover disjoint, increasing parts of the genome."""
    from bamqc_b200 import synth
    parts = []
    for lib_ in libs:
        rec, offs = synth.generate(genome, lib_)
        parts.append((rec[:int(offs[-1])], offs))
    records = np.concatenate([p for p, _ in parts] + [np.zeros(64, dtype=np.uint8)])
    offsets, base = [np.zeros(1, dtype=np.uint64)], 0
    for p, offs in parts:
        offsets.append(offs[1:] + np.uint64(base))
        base += p.size
    return records, np.concatenate(offsets)


def _rec_lanes(records, offsets, lane_ids):
    """Lane of every record (its RG:Z tag; the synthetic records carry it first among the tags of a known layout)."""
    out = []
    for i in range(len(offsets) - 1):
        r = bytes(records[int(offsets[i]):int(offsets[i + 1])])
        k = r.find(b"RGZ")
        out.append(lane_ids.index(r[k + 3:r.index(b"\0", k)].decode()) if k >= 0 else -1)
    return np.array(out)


def _pieces_vs_oracle(tmp_path, genome, header_lib, records, offsets, cuts, feed, klist=(32,), qlist=(17,)):
    """Cut the stream at the given fractions of its records, one engine per piece in shard mode (several submissions per
    piece), resolve the coverage windows per lane, merge, and compare with the oracle on the whole file."""
    from bamqc_b200 import Engine, synth, dist
    lane_ids = synth.lane_ids(header_lib)
    n = len(offsets) - 1
    fasta, bam = tmp_path / "g.fa", tmp_path / "whole.ubam"
    genome.write_fasta(fasta)
    synth.write_bam(bam, genome, header_lib, records, int(offsets[-1]))
    r = util.run_oracle(bam, fasta, tmp_path / "oracle.bamqc", chroms="chr1,chr2", klist=klist, qlist=qlist)
    assert r.returncode == 0, r.stderr
    bounds = [0] + [int(n * c) for c in cuts] + [n]
    engines = []
    try:
        for lo, hi in zip(bounds[:-1], bounds[1:]):
            e = Engine(lane_ids=lane_ids, ref_names=genome.names, chroms="chr1,chr2", klist=klist, qlist=qlist, staging_bytes=8 << 20)
            engines.append(e)
            for rid, (p, m) in enumerate(zip(genome.packed, genome.lengths)):
                e.set_reference(rid, p, m)
            e.cov_defer(2 if (lo == 0 and len(cuts) != 2) else 1)   # the first piece may run like a stand-alone engine
            step = max(1, (hi - lo) // 3)
            for a in range(lo, hi, step):
                b = min(hi, a + step)
                o = offsets[a:b + 1]
                if feed == "host":   # offsets given: the host finds every record's lane
                    e.submit(records[int(o[0]):int(o[-1])], o - o[0])
                elif feed == "device":   # whole records framed on the device, lanes from k_frame_lanes
                    e.submit(records[int(o[0]):int(o[-1])], None)
                else:   # the byte stream in arbitrary chunks
                    e.submit_stream(records[int(o[0]):int(o[-1])], last=b == hi)
            e.finish()
        deltas = dist.resolve_coverage_local_lanes(engines, len(lane_ids))
        assert len(deltas) == len(lane_ids)
        for e in engines[1:]:
            engines[0].merge_from(e)
        for lane, d in enumerate(deltas):
            engines[0].poscov_adjust(d, lane)
        engines[0].write_bamqc("S1", tmp_path / "merged.bamqc")
    finally:
        for e in engines:
            e.close()
    diffs = util.diff_bamqc(tmp_path / "oracle.bamqc", tmp_path / "merged.bamqc")
    assert not diffs, "\n".join(diffs)
    return bounds


@pytest.mark.parametrize("feed", ["host", "device", "stream"])
@pytest.mark.parametrize("cuts", CUTS)
def test_three_lanes_one_sorted_stream_cut_at_arbitrary_records(tmp_path, cuts, feed):
    from bamqc_b200 import synth
    genome = util.small_genome(seed=23, lengths=(300000, 200000, 50000))
    lib_ = synth.Library(seed=78, n_pairs=15000, n_lanes=3)
    records, offsets = synth.generate(genome, lib_)
    lanes = _rec_lanes(records, offsets, synth.lane_ids(lib_))
    assert set(lanes.tolist()) == {0, 1, 2}
    _pieces_vs_oracle(tmp_path, genome, lib_, records, offsets, cuts, feed)


def test_lane_only_in_the_first_third(tmp_path):
    """Lane L3 occurs in the first third of the file only: the later pieces hold none of its records."""
    from bamqc_b200 import synth
    genome = util.small_genome(seed=24, lengths=(400000, 300000, 100000))
    libs = [synth.Library(seed=530, n_pairs=4000, n_lanes=3, regions={0: (0, 400000)}, emit_unmapped_tail=0),
            synth.Library(seed=531, n_pairs=8000, n_lanes=2, regions={1: (0, 300000)}, first_pair_id=10 ** 6)]
    records, offsets = _concat(genome, libs)
    lanes = _rec_lanes(records, offsets, synth.lane_ids(libs[0]))
    n = len(offsets) - 1
    last3 = int(np.nonzero(lanes == 2)[0].max())
    assert last3 < n // 2
    bounds = _pieces_vs_oracle(tmp_path, genome, libs[0], records, offsets, (0.5, 0.8), "device")
    assert bounds[1] > last3


def test_lane_without_records_and_lane_off_the_chromosome_set(tmp_path):
    """The header lists four lanes.  L4 has no record at all; L3 has records only on chrX (not in -c) and among the
    unmapped reads at the end, so no record of it takes part in the coverage statistic."""
    from bamqc_b200 import synth
    genome = util.small_genome(seed=25, lengths=(400000, 300000, 100000))
    libs = [synth.Library(seed=540, n_pairs=6000, n_lanes=2, regions={0: (0, 400000), 1: (0, 300000)}, emit_unmapped_tail=0),
            synth.Library(seed=541, n_pairs=3000, n_lanes=3, regions={2: (0, 100000)}, first_pair_id=10 ** 6)]
    records, offsets = _concat(genome, libs)
    header = synth.Library(n_lanes=4)
    lanes = _rec_lanes(records, offsets, synth.lane_ids(header))
    assert 3 not in set(lanes.tolist()) and 2 in set(lanes.tolist())
    _pieces_vs_oracle(tmp_path, genome, header, records, offsets, (0.3, 0.6, 0.9), "host")


def test_two_lanes_several_q_and_k(tmp_path):
    """-k 15,32,63 -q 10,17: the per-lane sketches of two pieces merge."""
    from bamqc_b200 import synth
    genome = util.small_genome(seed=26, lengths=(300000, 200000, 50000))
    lib_ = synth.Library(seed=79, n_pairs=8000, n_lanes=2)
    records, offsets = synth.generate(genome, lib_)
    _pieces_vs_oracle(tmp_path, genome, lib_, records, offsets, (0.45,), "device", klist=(15, 32, 63), qlist=(10, 17))


@pytest.fixture(scope="module")
def multi_rg_bgzf(tmp_path_factory):
    """A three-lane level-1 BGZF file of more than 12 MB (every piece of a 3-way cut gets the command's 4 MB minimum)
    and the oracle's .bamqc of it."""
    from bamqc_b200 import synth
    d = tmp_path_factory.mktemp("lanes_cli")
    genome = util.small_genome(seed=27, lengths=(400000, 300000, 100000))
    lib_ = synth.Library(seed=550, n_pairs=85000, n_lanes=3)
    records, offsets = synth.generate(genome, lib_)
    n = int(offsets[-1])
    fasta, ubam, bam = d / "g.fa", d / "whole.ubam", d / "whole.bam"
    genome.write_fasta(fasta)
    synth.write_bam(ubam, genome, lib_, records, n)
    synth.write_bam(bam, genome, lib_, records, n, level=1)
    assert os.path.getsize(bam) >= 12 << 20
    r = util.run_oracle(ubam, fasta, d / "oracle.bamqc", chroms="chr1,chr2")
    assert r.returncode == 0, r.stderr
    return d, fasta, bam


@pytest.mark.parametrize("devices", ["0,0", "0,0,0", "0,1"])
def test_cli_devices_multi_read_group_bgzf(tmp_path, multi_rg_bgzf, devices):
    import torch
    d, fasta, bam = multi_rg_bgzf
    if len(set(devices.split(","))) > torch.cuda.device_count():
        pytest.skip("needs %d GPUs" % len(set(devices.split(","))))
    g = util.run_cli(["-r", fasta, "-c", "chr1,chr2", "-o", tmp_path / "gpu.bamqc", "--timing", "--devices", devices, bam])
    assert g.returncode == 0, g.stderr + g.stdout
    n = len(devices.split(","))
    assert ("devices=%d" % n) in g.stderr and "could not be cut" not in g.stderr, g.stderr
    diffs = util.diff_bamqc(d / "oracle.bamqc", tmp_path / "gpu.bamqc")
    assert not diffs, "\n".join(diffs)
