#!/usr/bin/env python3
"""Digests of the CPU oracle's output on the repeat-rich data sets and option sets of the two live comparisons with the
reference in tests/test_oracle_vs_golden.py (test_oracle_matches_live_reference_on_repeats and
test_oracle_dp_fallback_matches_live_reference), written to tests/golden/repeats.oracle.json.

These are the ORACLE's outputs (oracle/pbsc_oracle at the commit that wrote the file), not the reference's: they pin what the
oracle, the checker of the GPU tests, writes on these inputs, so a change to it shows in the CPU suite. The comparison with the
reference itself stays live and needs oracle/_ref/stride.  The index is built by bwt_build (byte-identical to `stride index`,
test_host_side).

    python tests/golden/make_repeats_golden.py
"""
import hashlib
import json
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
OUT = os.path.join(HERE, "repeats.oracle.json")

# name: (genome seed, coverage, read seed, pbcorrect options) -- as in the two live tests
CASES = {
    "nodp_c45": (21, 45, 211, ["-c", "45", "-g", "5", "--nodp"]),
    "nodp_c70_split": (21, 45, 211, ["-c", "70", "-g", "10", "--nodp", "--split"]),
    "nodp_c45_n3_m2": (21, 45, 211, ["-c", "45", "-g", "5", "--nodp", "-n", "3", "-m", "2"]),
    "dp_45x_c45": (23, 45, 213, ["-c", "45", "-g", "5"]),
    "dp_45x_c70_split_n2": (23, 45, 213, ["-c", "70", "-g", "10", "--split", "-n", "2"]),
    "dp_9x_c30": (23, 9, 213, ["-c", "30", "-g", "5"]),
    "dp_9x_c30_split": (23, 9, 213, ["-c", "30", "-g", "5", "--split"]),
}


def summary(text):
    return "\n".join(l for l in text.splitlines() if not l.startswith("Time of")).strip()


def digests(oracle_bin, workdir, name):
    """Run the oracle on one case in `workdir`; sha256 of each output file and of the summary block."""
    sys.path.insert(0, ROOT)
    from longreadselfcorrect_b200 import bwt_build, synth
    gseed, cov, rseed, opts = CASES[name]
    g = synth.make_genome(15000, gseed, repeat_families=1, tandem_arrays=3)
    codes, off = synth.simulate_reads(g, cov, 1200, rseed, min_len=300)
    reads = os.path.join(workdir, "reads.fa")
    synth.write_fasta(reads, codes, off)
    prefix = os.path.join(workdir, "idx")
    bwt_build.build_index_files(prefix, codes, off, device="cpu")
    out = os.path.join(workdir, "out")
    r = subprocess.run([oracle_bin, "pbcorrect", "--threads", "4", "-p", prefix, "-o", out] + opts + [reads], check=True,
                       stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    res = {f: hashlib.sha256(open(os.path.join(out, f), "rb").read()).hexdigest() for f in ("correct.fa", "discard.fa", "threshold-table")}
    res["summary"] = summary(r.stdout)
    return res


def main():
    import tempfile
    oracle_bin = os.path.join(ROOT, "oracle", "pbsc_oracle")
    res = {}
    for name in CASES:
        with tempfile.TemporaryDirectory() as d:
            res[name] = digests(oracle_bin, d, name)
    with open(OUT, "w") as f:
        json.dump(res, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
