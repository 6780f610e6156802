"""CPU check of the device SAM grammar (bamqc_b200/csrc/sam_parse.h): on random, deliberately odd lines every line it
accepts encodes byte for byte like the host encoder sam_line_to_bam (sam_text.h), and every line the host would encode
differently or reject is refused."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_fast_lines_encode_like_the_host_encoder(tmp_path):
    exe = str(tmp_path / "sam_selftest")
    subprocess.run(["g++", "-O2", "-std=c++17", "-o", exe, os.path.join(ROOT, "tests", "sam_selftest.cpp")], check=True)
    r = subprocess.run([exe, "200000"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert " 0 mismatching" in r.stdout
    fast, slow = (int(r.stdout.split(" fast")[0].split()[-1]), int(r.stdout.split(" not fast")[0].split()[-1]))
    assert fast > 20000 and slow > 20000, r.stdout   # both sides of the grammar are exercised


def test_parse_sam_header():
    from bamqc_b200 import parse_sam_header
    text = "@HD\tVN:1.6\r\n@SQ\tSN:chr1\tLN:1000\n@SQ\tSN:chr2\tLN:500\n@RG\tID:L1\tSM:S7\n@RG\tID:L2\tSM:S8\nr1\t0\tchr1\t1\n"
    h, used = parse_sam_header(text)
    assert used == text.index("\nr1\t") + 1
    assert h["ref_names"] == ["chr1", "chr2"] and h["ref_lengths"] == [1000, 500]
    assert h["lane_ids"] == ["L1", "L2"] and h["sample_id"] == "S8"
    assert "\r" not in h["text"]
