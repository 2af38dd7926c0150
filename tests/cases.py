"""Shared parity-test cases: deterministic inputs + runners for the oracle and the CUDA engine.

A case is a dict: contigs [(name, length, ref_bytes, win_beg)], batch (all reads, file order),
regions [(contig_index, beg1, end1)] in 1-based inclusive coordinates as a user would write
them, ``site_list`` (True: -l loop, False: argv regions), flags, lib_names.
"""
from __future__ import annotations

import gzip
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from bam_readcount_b200 import synth  # noqa: E402
from bam_readcount_b200.batch import BatchBuilder, ReadBatch  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")

FLAG_SETS = {
    "default": dict(),
    "q20b20": dict(min_mapq=20, min_bq=20),
    "ic": dict(insertion_centric=True),
    "perlib": dict(per_lib=True),
    "perlib_ic_q20b20": dict(per_lib=True, insertion_centric=True, min_mapq=20, min_bq=20),
    "d5": dict(max_cnt=5),
}


def flags_to_argv(fl: dict) -> list:
    a = []
    if "min_mapq" in fl:
        a += ["-q", str(fl["min_mapq"])]
    if "min_bq" in fl:
        a += ["-b", str(fl["min_bq"])]
    if "max_cnt" in fl:
        a += ["-d", str(fl["max_cnt"])]
    if fl.get("per_lib"):
        a += ["-p"]
    if fl.get("insertion_centric"):
        a += ["-i"]
    return a


def synthetic_case(L=30000, depth=30, seed=7, regions=((0, 3000, 23000),), site_list=False, n_libs=8):
    ref = synth.synth_reference(L, seed)
    batch = synth.synth_reads(ref, depth, seed=seed, n_libs=n_libs)
    return dict(name=f"syn_L{L}_d{depth}_s{seed}", contigs=[("chr1", L, ref.tobytes(), 0)], batch=batch,
                regions=list(regions), site_list=site_list, lib_names=[f"lib{i}" for i in range(n_libs)])


def deep_case(n_sites=3, depth=5000, seed=5, n_libs=8, L=2000):
    ref = synth.synth_reference(L, seed)
    sites = np.linspace(400, L - 400, n_sites).astype(np.int64)
    batch, bounds = synth.synth_deep_panel(ref, sites, depth, seed=seed, n_libs=n_libs)
    # one BAM: merge all groups and sort by position (stable) like a coordinate-sorted file
    order = np.argsort(batch.pos, kind="stable")
    batch = batch.select(order)
    return dict(name=f"deep_{n_sites}x{depth}", contigs=[("chr1", L, ref.tobytes(), 0)], batch=batch,
                regions=[(0, int(s) + 1, int(s) + 1) for s in sites], site_list=True,
                lib_names=[f"lib{i}" for i in range(n_libs)])


def testbam_case(bad_rg=False):
    """The reference's own fixture (R:test-data/test.bam + site_list), stored decoded under tests/golden/."""
    z = np.load(os.path.join(GOLDEN, "test_bam_bad_rg.npz" if bad_rg else "test_bam.npz"), allow_pickle=False)
    batch = ReadBatch(**{k: z[k] for k in ("tid", "pos", "flag", "mapq", "lib", "l_qseq", "nm", "sm", "cigar_off", "cigar",
                                           "seq_off", "seq", "qual_off", "qual")})
    win_beg = int(z["ref_win_beg"])
    ref = z["ref_win"].tobytes()
    return dict(name="test_bam_bad_rg" if bad_rg else "test_bam", contigs=[("21", int(z["chrom_len"]), ref, win_beg)],
                tid_map={20: 0}, batch=batch, regions=[(0, 10402985, 10402985), (0, 10405200, 10405200)], site_list=True,
                lib_names=[s for s in str(z["lib_names"]).split("\t") if s])


def case_tid(case, ci):
    """BAM tid of contig index ci (the goldens' contig 21 has tid 20 in test.bam)."""
    inv = {v: k for k, v in case.get("tid_map", {}).items()}
    return inv.get(ci, ci)


def region_reads(case, ci, beg1, end1):
    """Records the index iterator yields for samfetch(d.beg-1, d.end) (R:bamreadcount.cpp:602)."""
    beg, end = beg1 - 1, end1
    tid = case_tid(case, ci)
    idx = case["batch"].fetch(tid, beg - 1, end)
    return tid, beg, end, case["batch"].select(idx)


def run_oracle(case, flags, site_list=None):
    from oracle.oracle import Oracle
    sl = case["site_list"] if site_list is None else site_list
    o = Oracle(lib_names=case["lib_names"], **flags)
    for (ci, b1, e1) in case["regions"]:
        name, clen, seq, wb = case["contigs"][ci]
        tid, beg, end, sub = region_reads(case, ci, b1, e1)
        o.region(sub, tid=tid, beg=beg, end=end, contig=name, chrom_len=clen, ref_seq=seq, ref_win_beg=wb, site_list_mode=sl)
    return o.text(), o.dump(), o.warnings()


def run_engine(case, flags, site_list=None, want_dump=True):
    from bam_readcount_b200.engine import Engine, admitted
    sl = case["site_list"] if site_list is None else site_list
    e = Engine(lib_names=case["lib_names"], **flags)
    try:
        refs = {}
        for ci, (name, clen, seq, wb) in enumerate(case["contigs"]):
            tid = case_tid(case, ci)
            e.set_reference(tid, name, clen, seq, wb)
            refs[tid] = (wb, seq)
        pushed = []
        for (ci, b1, e1) in case["regions"]:
            tid, beg, end, sub = region_reads(case, ci, b1, e1)
            e.begin_region(tid, beg, end, sl)
            e.push_reads(sub)
            e.end_region()
            if want_dump:
                pushed.append(sub.select(admitted(sub, tid, flags.get("max_cnt", 10_000_000))))
        res = e.compute()
        text = e.format_text(-1)
        dump = res.dump(ReadBatch.concat(pushed), refs) if want_dump and pushed else ""
        warn = e.warnings()
        timing = (e.stage_ms(0), e.stage_ms(1))
        return text, dump, warn, timing
    finally:
        e.close()


def load_golden_text(name: str) -> str:
    p = os.path.join(GOLDEN, name)
    if os.path.exists(p + ".gz"):
        with gzip.open(p + ".gz", "rb") as fh:
            return fh.read().decode("latin-1")
    with open(p, "rb") as fh:
        return fh.read().decode("latin-1")


def assert_reference_output(key: str, stdout: bytes, stderr: bytes = None) -> None:
    """``stdout`` (and ``stderr``) equal what the reference binary printed for the test case ``key``: its exit code, line counts
    and SHA-256 digests are stored in tests/golden/reference_outputs.json (tests/golden/make_reference_outputs.py)."""
    with open(os.path.join(GOLDEN, "reference_outputs.json")) as fh:
        want = json.load(fh)[key]
    assert want["rc"] == 0, key
    assert (stdout.count(b"\n"), hashlib.sha256(stdout).hexdigest()) == (want["stdout_lines"], want["stdout_sha256"]), key
    if stderr is not None:
        assert (stderr.count(b"\n"), hashlib.sha256(stderr).hexdigest()) == (want["stderr_lines"], want["stderr_sha256"]), key
