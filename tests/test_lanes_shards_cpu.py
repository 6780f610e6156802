"""The per-lane coverage shard protocol of dist (resolve_coverage_shards_lanes) on CPU, world 2 and 3 over gloo, with a
mock engine of three lanes that differ: lane 0 plays back the pieces dumped by tests/cov_selftest.cpp (--dump-shards),
lane 1 is empty in every piece, lane 2 holds piece 0 only.  Each lane's correction must be bqc_cov_shards_combine of
that lane's own pieces, and the lanes must share the protocol's three exchanges."""
import ctypes
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_LANES = 3


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _empty_piece():
    return dict(n=0, first_rid=0, first_b=0, last_rid=0, last_b=0, table=list(range(1002)), span=0, head=[0] * 2001, tail=[0] * 2001)


def _lane_pieces(dump, world):
    """[lane][piece] -> the piece as the engine of that piece answers for that lane."""
    full = dump["pieces"]
    return [full, [_empty_piece() for _ in range(world)], [full[0]] + [_empty_piece() for _ in range(world - 1)]]


class _MockLaneEngine:
    """What an engine in shard mode with several lanes answers for one piece; checks that every lane's calls get that
    lane's predecessor and entry state."""

    def __init__(self, pieces):
        from bamqc_b200 import _lib
        self.pieces = pieces   # [lane] -> piece dict
        self.lib = _lib.load_library()   # bqc_cov_shards_combine / bqc_cov_apply are host code: no GPU needed

    def cov_shard_boundary(self, lane=0):
        return _shard_of(self.pieces[lane], run=False)

    def cov_shard_function(self, have_prev, prev_rid, prev_b, lane=0):
        p = self.pieces[lane]
        if p["n"]:
            assert have_prev == p["have_prev"], lane
            if have_prev:
                assert (prev_rid, prev_b) == (p["prev_rid"], p["prev_b"]), lane
        return np.array(p["table"], dtype=np.uint16)

    def cov_shard_run(self, have_prev, prev_rid, prev_b, p_in, lane=0):
        p = self.pieces[lane]
        if p["n"]:
            assert p_in == p["p_in"], (lane, p_in, p["p_in"])
        return _shard_of(p)


def _shard_of(p, run=True):
    """The bqc_cov_shard a piece answers: boundary fields, plus span/head/tail once it has run."""
    from bamqc_b200 import _lib
    sh = _lib.bqc_cov_shard()
    sh.n, sh.first_rid, sh.first_b, sh.last_rid, sh.last_b = (p[k] for k in ("n", "first_rid", "first_b", "last_rid", "last_b"))
    if run:
        sh.span = p["span"]
        for i in range(2001):
            sh.head[i] = p["head"][i]
            sh.tail[i] = p["tail"][i]
    return sh


def _combine_lane(pieces):
    """bqc_cov_shards_combine on one lane's pieces, straight through the C ABI."""
    from bamqc_b200 import _lib
    arr = (_lib.bqc_cov_shard * len(pieces))(*[_shard_of(p) for p in pieces])
    delta = np.zeros(101, dtype=np.int64)
    _lib.load_library().bqc_cov_shards_combine(ctypes.cast(arr, ctypes.c_void_p), len(pieces), delta.ctypes.data)
    return delta


def _dump(tmp_path, world):
    exe = str(tmp_path / "cov_selftest")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "cov_selftest.cpp")], check=True)
    path = str(tmp_path / "shards.json")
    subprocess.run([exe, "--dump-shards", str(world), path], check=True)
    return path


def _worker(rank, world, port, dump_path, out_dir):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from bamqc_b200 import dist as bdist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lanes = _lane_pieces(json.load(open(dump_path)), world)
    eng = _MockLaneEngine([lanes[l][rank] for l in range(N_LANES)])
    inner = bdist.torch_exchange()
    calls = [0]

    def exchange(a):
        calls[0] += 1
        return inner(a)
    deltas = bdist.resolve_coverage_shards_lanes(eng, rank, exchange, N_LANES)
    np.savez(os.path.join(out_dir, f"r{rank}.npz"), deltas=np.stack(deltas), calls=calls[0])
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 3])
def test_lanes_shard_protocol_over_gloo(tmp_path, world):
    import torch.multiprocessing as mp
    dump = _dump(tmp_path, world)
    port = _free_port()
    mp.spawn(_worker, args=(world, port, dump, str(tmp_path)), nprocs=world, join=True)
    d = json.load(open(dump))
    lanes = _lane_pieces(d, world)
    want = [_combine_lane(lanes[l]) for l in range(N_LANES)]
    assert not np.array_equal(want[0], want[1]) and not np.array_equal(want[0], want[2]) and not np.array_equal(want[1], want[2])
    total = np.sum([np.array(p["poscov"], dtype=np.int64) for p in d["pieces"]], axis=0)
    for r in range(world):
        got = np.load(tmp_path / f"r{r}.npz")
        assert int(got["calls"]) == 3
        assert got["deltas"].shape == (N_LANES, 101)
        for lane in range(N_LANES):
            assert np.array_equal(got["deltas"][lane], want[lane]), lane
        assert np.array_equal(total + got["deltas"][0], np.array(d["expected"], dtype=np.int64))


def test_lanes_shard_protocol_in_one_process(tmp_path):
    """dist.resolve_coverage_local_lanes: the same protocol for engines that live in one process."""
    from bamqc_b200 import dist as bdist
    world = 3
    lanes = _lane_pieces(json.load(open(_dump(tmp_path, world))), world)
    engines = [_MockLaneEngine([lanes[l][k] for l in range(N_LANES)]) for k in range(world)]
    deltas = bdist.resolve_coverage_local_lanes(engines, N_LANES)
    for lane in range(N_LANES):
        assert np.array_equal(deltas[lane], _combine_lane(lanes[lane])), lane
