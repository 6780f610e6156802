"""k_sketch32v2 hashes only the pieces of a read that end a window of 32 valid bases, spread over the warp, and walks
whole reads when that would not be shorter.  Every v2 instantiation (BQC_SKETCH_V2=1..4) against the CPU oracle -- the
`.bamqc` text, and the raw sketch, F2 table and sumCount of every (lane, q, k) -- at quality cutoffs whose share of
valid windows is 0 (stress library, -q 17), about 1 % (stress, -q 3), about 10 % (-q 17), about 50 % (-q 3) and 100 %
(-q 2), for 2 x 150, 2 x 700 and 2 x 1500 bp reads."""
import pytest

from test_dispatch_gpu import _parity
import bqc_testutil as util

pytestmark = pytest.mark.gpu

V2_KERNEL = {1: "k_sketch32v2<1024u>", 2: "k_sketch32v2<512u>", 3: "k_sketch32v2<640u>", 4: "k_sketch32v2<768u>"}


@pytest.mark.parametrize("v2", [1, 2, 3, 4])
def test_sketch_pieces_quality_profiles(tmp_path, monkeypatch, v2):
    from bamqc_b200 import synth
    monkeypatch.setenv("BQC_SKETCH_V2", str(v2))
    names = _parity(tmp_path / "std", synth.Library(seed=700 + v2, n_pairs=4000), qlist=(2, 3, 17), mutate=False)
    util.assert_kernels(names, (V2_KERNEL[v2],))
    names = _parity(tmp_path / "stress", synth.Library(seed=710 + v2, n_pairs=4000).stress(), qlist=(3, 17), mutate=False,
                    extra_short=False)
    util.assert_kernels(names, (V2_KERNEL[v2],))


@pytest.mark.parametrize("v2", [1, 2, 3, 4])
def test_sketch_pieces_long_reads(tmp_path, monkeypatch, v2):
    from bamqc_b200 import synth
    monkeypatch.setenv("BQC_SKETCH_V2", str(v2))
    lib700 = synth.Library(seed=720 + v2, n_pairs=800, read_len=700, ins_mean=1200, ins_sd=100, ins_min=800, ins_max=2000)
    names = _parity(tmp_path / "r700", lib700, qlist=(2, 17, 30), isize=3000, extra_short=False)
    util.assert_kernels(names, (V2_KERNEL[v2],))
    lib1500 = synth.Library(seed=730 + v2, n_pairs=300, read_len=1500, ins_mean=2500, ins_sd=100, ins_min=1800, ins_max=4000)
    names = _parity(tmp_path / "r1500", lib1500, qlist=(2, 17, 30), isize=3000, extra_short=False)
    util.assert_kernels(names, (V2_KERNEL[v2],))
