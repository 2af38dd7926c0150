"""The C++ host `brc-readcount`: same command line and STDOUT as bam-readcount.
CPU: flag handling that needs no device.  GPU: the reference's six integration-test command lines
(R:integration-test/bam-readcount_test.py:29-116) against its golden files, through BGZF/BAM/BAI/FASTA
decode -> C ABI -> CUDA kernels -> text emitter."""
import os
import subprocess

import numpy as np
import pytest

import bamwrite
import cases

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _cli():
    from bam_readcount_b200 import build
    build.build()
    return build.build_cli()


def test_cli_help_and_version_exit_code_1():
    exe = _cli()
    for flag in ("-h", "-v"):
        p = subprocess.run([exe, flag], capture_output=True)
        assert p.returncode == 1          # R:src/exe/bam-readcount/bamreadcount.cpp:467-475
    p = subprocess.run([exe], capture_output=True)
    assert p.returncode == 1 and b"Usage: bam-readcount" in p.stdout


def _write_ref(tmp):
    """ref.fa of contig 21: N everywhere except the window the fixture reads touch (stored in test_bam.npz)."""
    z = np.load(os.path.join(GOLDEN, "test_bam.npz"))
    L, wb = int(z["chrom_len"]), int(z["ref_win_beg"])
    seq = np.full(L, ord("N"), dtype=np.uint8)
    seq[wb:wb + z["ref_win"].shape[0]] = z["ref_win"]
    from bam_readcount_b200 import synth
    synth.write_fasta(os.path.join(tmp, "ref.fa"), "21", seq)
    return os.path.join(tmp, "ref.fa")


@pytest.mark.gpu
@pytest.mark.parametrize("args,bam,golden", [
    (["-w", "1", "-l", "site_list"], "test.bam", "expected_all_lib"),
    (["-w", "1", "-p", "-l", "site_list"], "test.bam", "expected_per_lib"),
    (["-w", "1", "-i", "-l", "site_list"], "test.bam", "expected_insertion_centric_all_lib"),
    (["-w", "1", "-i", "-p", "-l", "site_list"], "test.bam", "expected_insertion_centric_per_lib"),
    (["-w", "1", "REGIONS"], "test.bam", "expected_all_lib"),
    (["-w", "1", "REGIONS"], "test_bad_rg.bam", "expected_all_lib"),
])
def test_cli_reproduces_reference_goldens(tmp_path, args, bam, golden):
    exe = _cli()
    ref = _write_ref(str(tmp_path))
    argv = [exe, "-f", ref]
    regions = []
    for a in args:
        if a == "REGIONS":
            regions = ["21:10402985-10402985", "21:10405200-10405200"]
        elif a == "site_list":
            argv.append(os.path.join(GOLDEN, "site_list"))
        else:
            argv.append(a)
    argv.append(os.path.join(GOLDEN, bam))
    argv += regions
    p = subprocess.run(argv, capture_output=True)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    assert p.stdout.decode("latin-1") == cases.load_golden_text(golden)
    assert b"Minimum mapping quality is set to 0" in p.stderr


@pytest.mark.gpu
def test_cli_synthetic_bam_matches_oracle(tmp_path):
    """A coordinate-sorted synthetic BAM (tests/bamwrite.py) through the CLI, whole-contig region and a site list, against the
    CPU oracle."""
    from bam_readcount_b200 import synth
    exe = _cli()
    case = cases.synthetic_case(L=40000, depth=30, seed=31, regions=((0, 1001, 38000),), site_list=False)
    name, L, seq, _ = case["contigs"][0]
    d = str(tmp_path)
    synth.write_fasta(os.path.join(d, "ref.fa"), name, np.frombuffer(seq, dtype=np.uint8))
    bamwrite.write_bam(os.path.join(d, "s.bam"), case["batch"], [(name, L)])
    for fl, argv in ((dict(min_mapq=20, min_bq=20), ["-q", "20", "-b", "20"]), (dict(per_lib=True, insertion_centric=True), ["-p", "-i"])):
        want, _, _ = cases.run_oracle(case, fl, site_list=False)
        p = subprocess.run([exe, "-w", "0", "-f", os.path.join(d, "ref.fa")] + argv + [os.path.join(d, "s.bam"), "chr1:1001-38000"], capture_output=True)
        assert p.returncode == 0, p.stderr.decode()[-2000:]
        assert p.stdout.decode("latin-1") == want


@pytest.mark.gpu
def test_cli_windowed_long_region_equals_unsplit(tmp_path):
    """brc-readcount cuts long regions into windows (bounded memory); the concatenation must equal the unsplit output,
    deletions across window edges included."""
    from bam_readcount_b200 import synth
    exe = _cli()
    case = cases.synthetic_case(L=30000, depth=30, seed=41, regions=((0, 1, 30000),), site_list=False)
    name, L, seq, _ = case["contigs"][0]
    d = str(tmp_path)
    synth.write_fasta(os.path.join(d, "ref.fa"), name, np.frombuffer(seq, dtype=np.uint8))
    bamwrite.write_bam(os.path.join(d, "s.bam"), case["batch"], [(name, L)])
    outs = []
    for win in ("100000000", "3777"):
        p = subprocess.run([exe, "-w", "0", "-p", "-f", os.path.join(d, "ref.fa"), os.path.join(d, "s.bam"), "chr1:1-30000"],
                           capture_output=True, env=dict(os.environ, BRC_CLI_WINDOW=win))
        assert p.returncode == 0, p.stderr.decode()[-2000:]
        outs.append(p.stdout)
    assert outs[0] == outs[1] and outs[0].count(b"\n") > 29000


def test_cli_bgzf_bai_region_fetch_matches_python_decoder(tmp_path):
    """CPU: the C++ host's BGZF (multi-threaded read-ahead) / BAM / BAI region fetch, checked against the Python decoder's
    linear scan: same records per region (count, sum of positions, sum of qualities)."""
    exe = _cli()
    from bam_readcount_b200.bamio import read_bam
    bam = os.path.join(GOLDEN, "test.bam")
    hdr, b = read_bam(bam)
    regions = [("21", 10402985, 10402985), ("21", 10405200, 10405200), ("21", 10402700, 10405300), ("21", 1, 10402000), ("21", 10403000, 10403100)]
    sl = tmp_path / "sites"
    sl.write_text("".join(f"{c}\t{s}\t{e}\n" for c, s, e in regions))
    p = subprocess.run([exe, "-l", str(sl), bam], capture_output=True, env=dict(os.environ, BRC_CLI_DECODE_ONLY="1", BRC_CLI_WINDOW="2000000000"))
    assert p.returncode == 0, p.stderr.decode()
    got = [tuple(int(x) for x in line.split("\t")) for line in p.stdout.decode().strip().splitlines()]
    assert len(got) == len(regions)
    qo = b.qual_off.astype(np.int64)
    for (c, s, e), g in zip(regions, got):
        tid = hdr.tid_of[c]
        idx = b.fetch(tid, s - 2, e)          # samfetch(d.beg-1, d.end) with d.beg = s-1
        want = (tid, s - 1, e, len(idx), int(b.pos[idx].astype(np.int64).sum()), int(sum(int(b.qual[qo[i]:qo[i + 1]].astype(np.int64).sum()) for i in idx)))
        assert g == want


def _site_list_regions(L, rng):
    """Sorted dense single sites, overlapping / nested / repeated regions, a backwards jump and far jumps."""
    regs = [(int(p), int(p)) for p in range(2000, 5500, 7)]
    regs += [(6000, 6400), (6100, 6150), (6100, 6150), (6149, 6700), (6700, 6700)]
    regs += [(3000, 3010)]                                     # backwards
    regs += [(int(p), int(p) + int(w)) for p, w in zip(np.sort(rng.integers(7000, L - 500, 150)), rng.integers(0, 40, 150))]
    regs += [(L - 300, L), (1, 50)]
    return regs


def _make_bam(case, d):
    from bam_readcount_b200 import synth
    name, L, seq, _ = case["contigs"][0]
    synth.write_fasta(os.path.join(d, "ref.fa"), name, np.frombuffer(seq, dtype=np.uint8))
    bamwrite.write_bam(os.path.join(d, "s.bam"), case["batch"], [(name, L)], n_libs=len(case["lib_names"]))
    return os.path.join(d, "s.bam"), os.path.join(d, "ref.fa")


def test_cli_site_list_fetch_merging_yields_samfetch_records(tmp_path):
    """CPU (SURVEY.md §8 f-3): consecutive site-list lines share one forward pass over the BAM instead of one index seek
    each; every region must still receive exactly the records samfetch yields.  Checked against the per-region seek path
    (BRC_CLI_NO_MERGE) and against the Python decoder."""
    exe = _cli()
    case = cases.synthetic_case(L=60000, depth=30, seed=77, regions=((0, 1, 60000),), site_list=True)
    bam, _ = _make_bam(case, str(tmp_path))
    regs = _site_list_regions(60000, np.random.default_rng(5))
    sl = tmp_path / "sites"
    sl.write_text("".join(f"chr1\t{s}\t{e}\n" for s, e in regs))
    outs, stats = [], []
    for extra in ({}, {"BRC_CLI_NO_MERGE": "1"}):
        p = subprocess.run([exe, "-l", str(sl), bam], capture_output=True, env=dict(os.environ, BRC_CLI_DECODE_ONLY="1", BRC_CLI_TIMING="1", **extra))
        assert p.returncode == 0, p.stderr.decode()
        outs.append(p.stdout.decode())
        line = [ln for ln in p.stderr.decode().splitlines() if "index seeks" in ln][0].split()
        stats.append((int(line[4]), int(line[7])))
    assert outs[0] == outs[1]
    assert stats[0][0] < 20 and stats[1][0] == len(regs)          # a handful of seeks instead of one per line
    assert stats[0][1] * 20 < stats[1][1]                          # and far fewer records decoded
    b = case["batch"]
    qo = b.qual_off.astype(np.int64)
    got = [tuple(int(x) for x in line.split("\t")) for line in outs[0].strip().splitlines()]
    for (s, e), g in zip(regs, got):
        idx = b.fetch(0, max(s - 2, 0), e)
        want = (0, s - 1, e, len(idx), int(b.pos[idx].astype(np.int64).sum()), int(sum(int(b.qual[qo[i]:qo[i + 1]].astype(np.int64).sum()) for i in idx)))
        assert g == want, (s, e)


@pytest.mark.gpu
def test_cli_dense_site_list_matches_oracle(tmp_path):
    """A few hundred site-list lines (dense, overlapping, nested, repeated, out of order) through the merged fetch, the
    engine and the emitter, against the CPU oracle run region by region like the reference's -l loop."""
    exe = _cli()
    regs = _site_list_regions(60000, np.random.default_rng(5))
    case = cases.synthetic_case(L=60000, depth=30, seed=77, regions=tuple((0, s, e) for s, e in regs), site_list=True)
    bam, ref = _make_bam(case, str(tmp_path))
    sl = tmp_path / "sites"
    sl.write_text("".join(f"chr1\t{s}\t{e}\n" for s, e in regs))
    for fl, argv in ((dict(min_mapq=20, min_bq=20), ["-q", "20", "-b", "20"]), (dict(per_lib=True), ["-p"])):
        want, _, _ = cases.run_oracle(case, fl, site_list=True)
        outs = []
        for extra in ({}, {"BRC_CLI_NO_MERGE": "1"}):
            p = subprocess.run([exe, "-w", "0", "-f", ref] + argv + ["-l", str(sl), bam], capture_output=True, env=dict(os.environ, **extra))
            assert p.returncode == 0, p.stderr.decode()[-2000:]
            outs.append(p.stdout.decode("latin-1"))
        assert outs[0] == outs[1]
        assert outs[0] == want


def test_cli_fetch_merging_two_contigs_unsorted_and_past_the_end(tmp_path):
    """CPU: the merged fetch across contig changes, lines that go backwards, duplicates, a line past the contig's last read
    and an unknown contig — record sets identical to the one-seek-per-line path and to the Python decoder."""
    import dataclasses
    from bam_readcount_b200.batch import ReadBatch
    exe = _cli()
    a = cases.synthetic_case(L=30000, depth=20, seed=3, regions=((0, 1, 30000),), site_list=True)["batch"]
    b = cases.synthetic_case(L=20000, depth=25, seed=4, regions=((0, 1, 20000),), site_list=True)["batch"]
    b = dataclasses.replace(b, tid=np.ones_like(b.tid))
    both = ReadBatch.concat([a, b])
    d = str(tmp_path)
    bamwrite.write_bam(os.path.join(d, "s.bam"), both, [("chrA", 30000), ("chrB", 20000)])
    lines = [("chrA", 100, 100), ("chrA", 101, 130), ("chrB", 5000, 5000), ("chrB", 5001, 5001), ("chrA", 120, 125), ("chrA", 120, 125),
             ("chrB", 19990, 25000), ("chrA", 29999, 30000), ("chrZ", 5, 6), ("chrB", 1, 1), ("chrB", 2, 2), ("chrB", 3, 400)]
    sl = tmp_path / "sites"
    sl.write_text("".join(f"{c}\t{s}\t{e}\n" for c, s, e in lines))
    outs = []
    for extra in ({}, {"BRC_CLI_NO_MERGE": "1"}):
        p = subprocess.run([exe, "-l", str(sl), os.path.join(d, "s.bam")], capture_output=True, env=dict(os.environ, BRC_CLI_DECODE_ONLY="1", **extra))
        assert p.returncode == 0, p.stderr.decode()
        outs.append(p.stdout.decode())
        assert b"chrZ not found in bam file" in p.stderr
    assert outs[0] == outs[1]
    got = [tuple(int(x) for x in ln.split("\t")) for ln in outs[0].strip().splitlines()]
    known = [ln for ln in lines if ln[0] != "chrZ"]
    assert len(got) == len(known)
    qo = both.qual_off.astype(np.int64)
    for (c, s, e), g in zip(known, got):
        tid = 0 if c == "chrA" else 1
        idx = both.fetch(tid, max(s - 2, 0), e)
        want = (tid, s - 1, e, len(idx), int(both.pos[idx].astype(np.int64).sum()), int(sum(int(both.qual[qo[i]:qo[i + 1]].astype(np.int64).sum()) for i in idx)))
        assert g == want, (c, s, e)


# ---- the boundary compiled INTO the reference: its own main(), option parsing, htslib readers and region loops, with
# ---- fetch_func / pileup_func / the pileup buffer replaced by the C ABI (oracle/patch_reference.py, INTEGRATION.md §2)
def _patched_reference():
    exe = os.path.join(ROOT, "oracle", "_ref", "bam-readcount-brc")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/bam-readcount-brc not built (oracle/build_patched_ref.sh, needs /root/reference)")
    return exe


def test_patched_reference_needs_a_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    exe = _patched_reference()
    data = os.path.join(ROOT, "oracle", "_ref", "test-data")
    p = subprocess.run([exe, "-w", "1", "-f", "ref.fa", "-l", "site_list", "test.bam"], cwd=data, capture_output=True)
    assert p.returncode == 1 and b"no usable CUDA device" in p.stderr and p.stdout == b""      # no CPU fallback behind the boundary


@pytest.mark.gpu
@pytest.mark.parametrize("args,bam,golden", [
    (["-w", "1", "-l", "site_list"], "test.bam", "expected_all_lib"),
    (["-w", "1", "-p", "-l", "site_list"], "test.bam", "expected_per_lib"),
    (["-w", "1", "-i", "-l", "site_list"], "test.bam", "expected_insertion_centric_all_lib"),
    (["-w", "1", "-i", "-p", "-l", "site_list"], "test.bam", "expected_insertion_centric_per_lib"),
    (["-w", "1", "REGIONS"], "test.bam", "expected_all_lib"),
    (["-w", "1", "REGIONS"], "test_bad_rg.bam", "expected_all_lib"),
])
def test_reference_main_through_the_c_abi_reproduces_goldens(args, bam, golden):
    """R:integration-test/bam-readcount_test.py:29-116 — the six command lines, run by the reference's own main()
    linked against libbrc_engine.so."""
    exe = _patched_reference()
    data = os.path.join(ROOT, "oracle", "_ref", "test-data")
    argv = [exe, "-f", "ref.fa"]
    regions = []
    for a in args:
        if a == "REGIONS":
            regions = ["21:10402985-10402985", "21:10405200-10405200"]
        else:
            argv.append(a)
    argv.append(bam)
    argv += regions
    p = subprocess.run(argv, cwd=data, capture_output=True)
    assert p.returncode == 0, p.stderr.decode()[-2000:]
    assert p.stdout.decode("latin-1") == cases.load_golden_text(golden)


@pytest.mark.gpu
def test_reference_main_through_the_c_abi_on_the_cram():
    """BASELINE config 2b on the CRAM itself: htslib (the reference's reader) decodes twolib.sorted.cram, the engine computes."""
    exe = _patched_reference()
    data = os.path.join(ROOT, "oracle", "_ref", "test-data")
    for extra, golden in ((["-p"], "ref_cram_twolib_perlib.txt"), ([], "ref_cram_twolib_alllib.txt")):
        p = subprocess.run([exe, "-w", "0"] + extra + ["-f", "rand1k.fa", "-l", "twolib_site_list.txt", "twolib.sorted.cram"], cwd=data, capture_output=True)
        assert p.returncode == 0, p.stderr.decode()[-2000:]
        assert p.stdout.decode("latin-1") == cases.load_golden_text(golden)


WARNING_CASES = [
    (["-w", "3", "-l", "site_list"], "test.bam"),
    (["-w", "2", "-p", "-l", "site_list"], "test_bad_rg.bam"),
    (["-w", "5", "-i", "REGION"], "test.bam"),
    (["-w", "0", "-l", "site_list"], "test.bam"),
    (["-w", "1", "-q", "30", "-b", "25", "REGION"], "test.bam"),
]
REGION_FORMS = [["21:10405200"], ["21:10402985-10402985", "21:10405200"], ["21:10,402,985-10,402,990"], ["21:10402985-"],
                ["21:10402985-10402985", "21"], ["21:-5"], ["21:10402985-10402986", "21:10402987-10402990"]]


def warning_key(args, bam):
    return "warnings " + " ".join(args + [bam])


def warning_argv(ref, args, bam):
    """The command line after the program name: -f ref, the options, the BAM, then the region if any."""
    argv = ["-f", ref]
    regions = []
    for a in args:
        if a == "REGION":
            regions = ["21:10402980-10402995"]
        elif a == "site_list":
            argv.append(os.path.join(GOLDEN, "site_list"))
        else:
            argv.append(a)
    return argv + [os.path.join(GOLDEN, bam)] + regions


@pytest.mark.gpu
@pytest.mark.parametrize("args,bam", WARNING_CASES)
def test_cli_warning_lines_match_the_reference_binary(tmp_path, args, bam):
    """STDERR parity: the per-read warning lines (R:src/lib/bamrc/ReadWarnings.hpp:39-50) name the same reads, in the same order,
    with the same "has been emitted N times" line, as the unmodified reference binary on the same command line (its STDOUT and
    STDERR are stored as digests in tests/golden/reference_outputs.json)."""
    exe = _cli()
    ref = _write_ref(str(tmp_path))
    p = subprocess.run([exe] + warning_argv(ref, args, bam), capture_output=True)
    assert p.returncode == 0, p.stderr.decode()[-1000:]
    cases.assert_reference_output(warning_key(args, bam), p.stdout, p.stderr)


@pytest.mark.gpu
def test_cli_region_forms_match_the_reference_binary(tmp_path):
    """bam_parse_region corner cases (ADVICE r1): an open end keeps the previous / default beg-end, thousands separators are
    accepted, "chr:-N" starts at the first base — STDOUT identical to the reference binary's (stored as a digest)."""
    exe = _cli()
    ref = _write_ref(str(tmp_path))
    bam = os.path.join(GOLDEN, "test.bam")
    for regions in REGION_FORMS:
        o = subprocess.run([exe, "-w", "0", "-f", ref, bam] + regions, capture_output=True)
        assert o.returncode == 0
        cases.assert_reference_output("region_forms " + " ".join(regions), o.stdout)


def test_cli_reports_truncated_bam(tmp_path):
    """A BAM cut in the middle of a BGZF block is a decode ERROR, not end of file: non-zero exit and a diagnostic (ADVICE r1)."""
    exe = _cli()
    src = open(os.path.join(GOLDEN, "test.bam"), "rb").read()
    cut = os.path.join(str(tmp_path), "cut.bam")
    open(cut, "wb").write(src[:60000])
    import shutil
    shutil.copy(os.path.join(GOLDEN, "test.bam.bai"), cut + ".bai")
    env = dict(os.environ, BRC_CLI_DECODE_ONLY="1")
    p = subprocess.run([exe, "-w", "0", cut, "21:10402000-10406000"], capture_output=True, env=env)
    assert p.returncode == 1 and b"truncated or corrupt" in p.stderr
    q = subprocess.run([exe, "-w", "0", os.path.join(GOLDEN, "test.bam"), "21:10402000-10406000"], capture_output=True, env=env)
    assert q.returncode == 0 and b"truncated" not in q.stderr


def _cram_fixture():
    d = os.path.join(ROOT, "oracle", "_ref", "test-data")
    if not os.path.exists(os.path.join(d, "twolib.sorted.cram")):
        pytest.skip("oracle/_ref/test-data not present")
    exe = _cli()
    if b"BRC_WITH_HTSLIB" not in open(exe, "rb").read() and not os.path.exists(os.path.join(ROOT, "bam_readcount_b200", "third_party", "htslib", "libhts.a")):
        pytest.skip("host built without htslib (tools/build_htslib.sh)")
    return exe, d


def test_cli_decodes_cram_through_htslib():
    """BASELINE config 2b input: twolib.sorted.cram is decoded by the host (htslib), no device needed for the decode itself."""
    exe, d = _cram_fixture()
    p = subprocess.run([exe, "-w", "0", "-f", "rand1k.fa", "-l", "twolib_site_list.txt", "twolib.sorted.cram"], cwd=d, capture_output=True,
                       env=dict(os.environ, BRC_CLI_DECODE_ONLY="1"))
    assert p.returncode == 0, p.stderr.decode()
    assert b"Expect library: reads1_lb in BAM" in p.stderr
    tid, beg, end, n, psum, qsum = p.stdout.decode().split()
    assert (tid, beg, end) == ("0", "49", "60") and int(n) >= 1 and int(qsum) == 255 * 60 * int(n)     # CRAM without qualities: 0xFF


@pytest.mark.gpu
def test_cli_cram_config_2b_matches_reference_output():
    """BASELINE config 2b on twolib.sorted.cram itself (R:test-data/cram_site_test.sh:1): -p and all-library output equal the
    committed output of the reference binary."""
    exe, d = _cram_fixture()
    for extra, golden in ((["-p"], "ref_cram_twolib_perlib.txt"), ([], "ref_cram_twolib_alllib.txt")):
        p = subprocess.run([exe, "-w", "0"] + extra + ["-f", "rand1k.fa", "-l", "twolib_site_list.txt", "twolib.sorted.cram"], cwd=d, capture_output=True)
        assert p.returncode == 0, p.stderr.decode()[-2000:]
        assert p.stdout.decode("latin-1") == cases.load_golden_text(golden)


def test_cli_shards_partition_the_regions(tmp_path):
    """--shard RANK/COUNT: the ranks' units are a partition of the windowed regions, in order (decode-only, no device)."""
    from bam_readcount_b200 import synth_cb
    exe = _cli()
    sp = synth_cb.Spec(seed=3, contig_len=1280 * 400)
    info = bamwrite.write_sample_bam(sp, 0, 0, 400, str(tmp_path))
    env = dict(os.environ, BRC_CLI_DECODE_ONLY="1", BRC_CLI_WINDOW="20000")
    whole = subprocess.run([exe, "-w", "0", info["bam"], "chr1:1001-400000", "chr1:420001-500000"], capture_output=True, env=env)
    assert whole.returncode == 0
    parts = []
    for r in range(3):
        p = subprocess.run([exe, "-w", "0", "--shard", f"{r}/3", info["bam"], "chr1:1001-400000", "chr1:420001-500000"], capture_output=True, env=env)
        assert p.returncode == 0, p.stderr.decode()
        parts.append(p.stdout)
    assert b"".join(parts) == whole.stdout and all(len(x) > 0 for x in parts)
    sizes = [sum(int(l.split()[3]) for l in x.decode().splitlines()) for x in parts]      # records fetched per shard
    assert max(sizes) < 1.35 * min(sizes)                                                   # BAI-weighted: about equal coverage


@pytest.mark.gpu
def test_cli_sharded_output_concatenates_to_the_unsharded_output(tmp_path):
    from bam_readcount_b200 import synth_cb
    exe = _cli()
    sp = synth_cb.Spec(seed=8, contig_len=1280 * 300)
    info = bamwrite.write_sample_bam(sp, 0, 0, 300, str(tmp_path))
    env = dict(os.environ, BRC_CLI_WINDOW="50000")
    args = ["-w", "0", "-i", "-f", info["fasta"], info["bam"], "chr1:2001-380000"]
    whole = subprocess.run([exe] + args, capture_output=True, env=env)
    assert whole.returncode == 0, whole.stderr.decode()[-1000:]
    multi = subprocess.run(["bash", os.path.join(ROOT, "tools", "brc_multi.sh"), "3"] + args, capture_output=True, env=dict(env, BRC_NDEV="1"))
    assert multi.returncode == 0, multi.stderr.decode()[-1000:]
    assert multi.stdout == whole.stdout and len(whole.stdout.splitlines()) == 378000


def test_cli_parallel_window_decode_yields_samfetch_records(tmp_path):
    """Big fetches are decoded by several threads over position sub-ranges (ParallelFetcher) and concatenated: record count,
    position sum and quality sum per region must equal the sequential reader's, whatever the thread count and window size
    (decode-only, no device)."""
    from bam_readcount_b200 import synth_cb
    exe = _cli()
    sp = synth_cb.Spec(seed=5, contig_len=1280 * 700)
    info = bamwrite.write_sample_bam(sp, 0, 0, 700, str(tmp_path))
    regions = ["chr1:1-896000", "chr1:100001-700000", "chr1:5-300", "chr1"]
    outs = []
    for extra in ({"BRC_CLI_SEQUENTIAL": "1"}, {}, {"BRC_CLI_DECODE_THREADS": "3"}, {"BRC_CLI_DECODE_THREADS": "16", "BRC_CLI_WINDOW": "300000"},
                  {"BRC_CLI_SEQUENTIAL": "1", "BRC_CLI_WINDOW": "300000"}):
        p = subprocess.run([exe, "-w", "0", info["bam"]] + regions, capture_output=True, env=dict(os.environ, BRC_CLI_DECODE_ONLY="1", BRC_CLI_TIMING="1", **extra))
        assert p.returncode == 0, p.stderr.decode()[-1000:]
        outs.append((p.stdout, p.stderr.decode()))
    assert outs[0][0] == outs[1][0] == outs[2][0] and outs[3][0] == outs[4][0]
    assert len(outs[0][0].splitlines()) == 4 and int(outs[0][0].split()[3]) > 170000
    assert "windows decoded by" in outs[1][1] and "(+ 0 records in 0 windows" in outs[0][1] and "(+ 0 records in 0 windows" not in outs[1][1]


@pytest.mark.gpu
def test_cli_parallel_window_decode_text_and_warnings_equal_sequential(tmp_path):
    """The parallel window path (one borrowed, page-locked batch per window, next window decoded ahead) against the record-by-record
    path: STDOUT and the per-read warning lines on STDERR must be identical, also when a window boundary falls inside the region."""
    from bam_readcount_b200 import synth
    from bam_readcount_b200.batch import TAG_ABSENT
    exe = _cli()
    case = cases.synthetic_case(L=300000, depth=12, seed=97, regions=((0, 1, 300000),), site_list=False)
    b = case["batch"]
    rng = np.random.default_rng(3)
    nm = np.array(b.nm, copy=True); nm[rng.choice(b.n_reads, 400, replace=False)] = TAG_ABSENT      # reads the reference warns about
    import dataclasses
    case["batch"] = dataclasses.replace(b, nm=nm)
    d = str(tmp_path)
    _make_bam(case, d)
    for args in (["-w", "0", "-i"], ["-p", "-q", "20", "-b", "20"], ["-w", "7", "-p"]):
        outs = []
        for extra in ({"BRC_CLI_SEQUENTIAL": "1"}, {}, {"BRC_CLI_DECODE_THREADS": "3", "BRC_CLI_WINDOW": "280000"}):
            p = subprocess.run([exe] + args + ["-f", os.path.join(d, "ref.fa"), os.path.join(d, "s.bam"), "chr1:1-300000", "chr1:1001-2000"],
                               capture_output=True, env=dict(os.environ, **extra))
            assert p.returncode == 0, p.stderr.decode()[-2000:]
            outs.append((p.stdout, p.stderr))
        assert outs[0][0] == outs[1][0] == outs[2][0] and outs[0][0].count(b"\n") > 299000
        assert outs[0][1] == outs[1][1] == outs[2][1]
        if args[1] != "0":
            assert b"WARNING: In read" in outs[0][1]


def test_cli_parallel_window_decode_two_contigs_unmapped_and_edges(tmp_path):
    """CPU: the parallel window decode on a two-contig BAM with placed-but-unmapped records, a fetch that starts inside a read,
    a fetch past the last read, a site-list line long enough to be cut into windows, and a contig without reads behind it:
    per-region (count, position sum, quality sum) identical to the sequential reader and to the Python decoder's samfetch."""
    import dataclasses
    from bam_readcount_b200.batch import ReadBatch
    exe = _cli()
    a = cases.synthetic_case(L=600000, depth=4, seed=31, regions=((0, 1, 600000),), site_list=False)["batch"]
    b = cases.synthetic_case(L=400000, depth=5, seed=32, regions=((0, 1, 400000),), site_list=False)["batch"]
    rng = np.random.default_rng(9)
    fa = np.array(a.flag, copy=True); fa[rng.choice(a.n_reads, 300, replace=False)] |= 4          # unmapped but placed (mate-anchored)
    a = dataclasses.replace(a, flag=fa)
    b = dataclasses.replace(b, tid=np.ones_like(b.tid))
    both = ReadBatch.concat([a, b])
    d = str(tmp_path)
    bamwrite.write_bam(os.path.join(d, "s.bam"), both, [("chrA", 600000), ("chrB", 400000), ("chrC", 300000)])
    lines = [("chrA", 1, 600000), ("chrA", 100077, 500000), ("chrB", 50, 399000), ("chrA", 300000, 300001), ("chrB", 120000, 400000),
             ("chrC", 1, 300000), ("chrA", 590000, 600000)]
    sl = tmp_path / "sites"
    sl.write_text("".join(f"{c}\t{s}\t{e}\n" for c, s, e in lines))
    outs = []
    for extra in ({"BRC_CLI_SEQUENTIAL": "1"}, {}, {"BRC_CLI_DECODE_THREADS": "5", "BRC_CLI_WINDOW": "270000"}, {"BRC_CLI_SEQUENTIAL": "1", "BRC_CLI_WINDOW": "270000"}):
        p = subprocess.run([exe, "-l", str(sl), os.path.join(d, "s.bam")], capture_output=True, env=dict(os.environ, BRC_CLI_DECODE_ONLY="1", BRC_CLI_TIMING="1", **extra))
        assert p.returncode == 0, p.stderr.decode()[-1500:]
        outs.append((p.stdout.decode(), p.stderr.decode()))
    assert outs[0][0] == outs[1][0] and outs[2][0] == outs[3][0]
    assert "(+ 0 records in 0 windows" not in outs[1][1] and "(+ 0 records in 0 windows" not in outs[2][1]
    got = [tuple(int(x) for x in ln.split("\t")) for ln in outs[0][0].strip().splitlines()]
    assert len(got) == len(lines)
    qo = both.qual_off.astype(np.int64)
    mapped = (both.flag & 4) == 0
    for (c, s, e), g in zip(lines, got):
        tid = {"chrA": 0, "chrB": 1, "chrC": 2}[c]
        idx = [i for i in both.fetch(tid, max(s - 2, 0), e) if mapped[i]]
        want = (tid, s - 1, e, len(idx), int(both.pos[idx].astype(np.int64).sum()) if idx else 0, int(sum(int(both.qual[qo[i]:qo[i + 1]].astype(np.int64).sum()) for i in idx)))
        assert g == want, (c, s, e, g, want)
    # the cut form prints one line per window: their sums are the uncut line's
    cut = [tuple(int(x) for x in ln.split("\t")) for ln in outs[2][0].strip().splitlines()]
    assert len(cut) > len(lines)
