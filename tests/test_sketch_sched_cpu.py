"""CPU check of bamqc_b200/csrc/sketch_sched.h (the pass-1 masks, the piece split and the restart/warm-up rule of
k_sketch32v2) against a per-base restatement of the k = 32 rolling hash on random reads."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_sketch_pieces_emit_the_per_base_hashes(tmp_path):
    exe = str(tmp_path / "sketch_sched_selftest")
    subprocess.run(["g++", "-O2", "-Wall", "-o", exe, os.path.join(ROOT, "tests", "sketch_sched_selftest.cpp")], check=True)
    r = subprocess.run([exe, "30000"], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert " 0 mismatching" in r.stdout
