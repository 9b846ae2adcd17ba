"""The read window of the thread-per-alignment DP (csrc/pbsc_dp_thread.cuh), compiled for the host: the fill over a 16-word ring
of the 2-bit read, refilled one sweep ahead as the kernel's 1024-base pass does it, against the fill over the whole read.  The
ring aborts on any read outside the sweep's window or of a slot not yet refilled for it; flag words, traceback start, final
column and the traceback itself must be identical, over bands above, through and below the matrix, both strands, homopolymer
and two-letter strings, queries of 1 to 4000 bases and reads at the length bound."""
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_ring_window_fill_matches_whole_read_bit_for_bit(tmp_path):
    exe = str(tmp_path / "t")
    subprocess.run(["/usr/bin/g++", "-O2", "-std=c++17", "-Wall", "-Wno-sign-compare", os.path.join(ROOT, "tests", "cpp", "test_dp_window.cpp"),
                    "-o", exe], check=True)
    r = subprocess.run([exe, "1500"], stdout=subprocess.PIPE, text=True)
    assert r.returncode == 0 and " failed 0" in r.stdout, r.stdout
    refills = int(r.stdout.split("refills ")[1].split()[0])
    widest = int(r.stdout.split("widest-window ")[1].split()[0])
    assert refills > 0 and widest == 15, r.stdout
