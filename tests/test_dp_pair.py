"""The paired-column fill of the thread-per-alignment DP (csrc/pbsc_dp_thread.cuh), compiled for the host, against the same
fill one column at a time: identical flag words, traceback start and final column, over every band placement of small
matrices, random forward / reverse-complement rows, sweeps past the 256-row circular array and 4000-base extremes."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_paired_fill_matches_scalar_fill_bit_for_bit(tmp_path):
    exe = str(tmp_path / "t")
    subprocess.run(["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-Wno-sign-compare", os.path.join(ROOT, "tests", "cpp", "test_dp_pair.cpp"),
                    "-o", exe], check=True)
    r = subprocess.run([exe, "3000"], stdout=subprocess.PIPE, text=True)
    assert r.returncode == 0 and " failed 0" in r.stdout, r.stdout
    paired = int(r.stdout.split("paired-columns ")[1].split()[0])
    assert paired > 0, r.stdout
