"""The masked first and last blocks of the paired-column fill (csrc/pbsc_dp_thread.cuh, fill_pair), compiled for the host,
against the same fill one column at a time over placements aimed at those blocks; the previous-column accessor checks that a
paired sweep changes no slot outside its second column's rows and stores at most one score outside its pair stores."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_masked_blocks_match_scalar_fill_and_store_only_their_rows(tmp_path):
    exe = str(tmp_path / "t")
    subprocess.run(["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-Wno-sign-compare",
                    os.path.join(ROOT, "tests", "cpp", "test_dp_pair_masked.cpp"), "-o", exe], check=True)
    r = subprocess.run([exe], stdout=subprocess.PIPE, text=True)
    assert r.returncode == 0, r.stdout
    assert " failed 0 bad-stores 0 sweeps-with-scalar-stores 0 " in r.stdout and " covered 1" in r.stdout, r.stdout
    sweeps = int(r.stdout.split("paired-sweeps ")[1].split()[0])
    assert sweeps >= 1000, r.stdout
