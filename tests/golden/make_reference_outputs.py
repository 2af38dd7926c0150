#!/usr/bin/env python
"""Regenerates tests/golden/reference_outputs.json: what the UNMODIFIED reference binary (oracle/_ref/bam-readcount, built by
oracle/build_ref.sh) prints for the command lines of the tests that compare with it, so that those comparisons run without it.

Each entry holds the SHA-256 and the line count of the reference's STDOUT (and of its STDERR where a test compares that too)
and its exit code.  The inputs are the tests' own: the committed test.bam fixtures with the FASTA the tests write, the fresh
fuzz cases of test_differential_fuzz.py and the generator's sample window of test_synth_stream.py, written to BAM by the
samtools the reference vendors (oracle/_ref/samtools), as the tests did when they ran the reference binary themselves.
"""
import hashlib
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import cases  # noqa: E402
import test_cli  # noqa: E402
import test_differential_fuzz  # noqa: E402
import test_synth_stream  # noqa: E402
from bam_readcount_b200 import synth, synth_cb  # noqa: E402
from oracle.oracle import REF_BIN, REF_SAMTOOLS  # noqa: E402

OUT = os.path.join(HERE, "reference_outputs.json")


def entry(p, with_stderr=False):
    e = {"rc": p.returncode, "stdout_sha256": hashlib.sha256(p.stdout).hexdigest(), "stdout_lines": p.stdout.count(b"\n")}
    if with_stderr:
        e.update(stderr_sha256=hashlib.sha256(p.stderr).hexdigest(), stderr_lines=p.stderr.count(b"\n"))
    return e


def run(argv, **kw):
    return subprocess.run([REF_BIN] + argv, capture_output=True, **kw)


def main():
    assert os.path.exists(REF_BIN) and os.path.exists(REF_SAMTOOLS), "run oracle/build_ref.sh first"
    out = {}
    with tempfile.TemporaryDirectory() as d:
        ref = test_cli._write_ref(d)
        for args, bam in test_cli.WARNING_CASES:
            out[test_cli.warning_key(args, bam)] = entry(run(test_cli.warning_argv(ref, args, bam)), with_stderr=True)
        bam = os.path.join(test_cli.GOLDEN, "test.bam")
        for regions in test_cli.REGION_FORMS:
            out["region_forms " + " ".join(regions)] = entry(run(["-w", "0", "-f", ref, bam] + regions))

    for seed in test_differential_fuzz.SEEDS:
        case = test_differential_fuzz._case(seed)
        name, L, seq, _ = case["contigs"][0]
        with tempfile.TemporaryDirectory() as d:
            synth.write_fasta(os.path.join(d, "ref.fa"), name, np.frombuffer(seq, dtype=np.uint8))
            synth.write_sam(os.path.join(d, "s.sam"), case["batch"], [(name, L)], n_libs=len(case["lib_names"]))
            subprocess.check_call([REF_SAMTOOLS, "view", "-b", "-o", os.path.join(d, "s.bam"), os.path.join(d, "s.sam")])
            subprocess.check_call([REF_SAMTOOLS, "index", os.path.join(d, "s.bam")])
            with open(os.path.join(d, "sites"), "w") as fh:
                for (_, b1, e1) in case["regions"]:
                    fh.write(f"{name}\t{b1}\t{e1}\n")
            for fname, fl in case["flag_sets"].items():
                p = run(["-w", "0", "-f", os.path.join(d, "ref.fa")] + cases.flags_to_argv(fl) +
                        ["-l", os.path.join(d, "sites"), os.path.join(d, "s.bam")])
                out[f"fuzz {seed} {fname}"] = entry(p)

    sp, blocks, beg, end = test_synth_stream.SAMPLE
    with tempfile.TemporaryDirectory() as d:
        info = synth_cb.write_sample_bam(sp, 0, 0, blocks, d, REF_SAMTOOLS)
        for argv, _ in test_synth_stream.SAMPLE_FLAGS:
            out["synth_sample " + " ".join(argv)] = entry(run(["-w", "0"] + argv + ["-f", info["fasta"], info["bam"], f"chr1:{beg + 1}-{end}"]))

    with open(OUT, "w") as fh:
        json.dump(out, fh, indent=1, sort_keys=True)
        fh.write("\n")
    print(f"{OUT}: {len(out)} entries")


if __name__ == "__main__":
    main()
