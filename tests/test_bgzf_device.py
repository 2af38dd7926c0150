"""SURVEY.md §8 f-2: BGZF inflate + BAM framing on the device (bam_readcount_b200/csrc/brc_bgzf.cu).

CPU: the DEFLATE core the kernel runs (brc_bgzf.cuh, host+device code) against zlib on every block of the fixtures, and the BAI
span builder.  GPU: the device-decoded batch equals the host decoder's records field for field, and a region computed from the
compressed span equals the region computed from host-decoded reads (text and raw accumulators)."""
import os
import subprocess
import tempfile

import numpy as np
import pytest

import bamwrite
import cases
from bam_readcount_b200 import bamio

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

HARNESS = r'''
#include <cstdio>
#include <cstring>
#include <vector>
#include <zlib.h>
#include "brc_bgzf.cuh"
int main(int argc, char **argv) {
    int bad = 0, nblk = 0;
    for (int a = 1; a < argc; ++a) {
        FILE *f = fopen(argv[a], "rb"); std::vector<uint8_t> d; uint8_t buf[65536]; size_t n;
        while ((n = fread(buf, 1, sizeof buf, f)) > 0) d.insert(d.end(), buf, buf + n);
        fclose(f);
        size_t o = 0; static brc::inflate::Tables T;
        while (o + 18 <= d.size()) {
            const uint8_t *h = &d[o]; if (h[0] != 31 || h[1] != 139) break;
            size_t xlen = h[10] | (h[11] << 8); int bsize = -1;
            for (size_t i = 0; i + 4 <= xlen;) { size_t sl = h[12 + i + 2] | (h[12 + i + 3] << 8); if (h[12 + i] == 'B' && h[12 + i + 1] == 'C') bsize = h[12 + i + 4] | (h[12 + i + 5] << 8); i += 4 + sl; }
            size_t total = bsize + 1, hdr = 12 + xlen; const uint8_t *tail = h + total - 4;
            uint32_t isize = tail[0] | (tail[1] << 8) | (tail[2] << 16) | ((uint32_t)tail[3] << 24);
            std::vector<uint8_t> want(isize + 1), got(isize + 1);
            z_stream zs{}; inflateInit2(&zs, -15); zs.next_in = (Bytef *)h + hdr; zs.avail_in = total - hdr - 8; zs.next_out = want.data(); zs.avail_out = isize;
            int rc = inflate(&zs, Z_FINISH); inflateEnd(&zs);
            int r = brc::inflate::inflate_block(brc::inflate::Lanes{0, 1}, h + hdr, total - hdr - 8, got.data(), isize, T);
            if (r != 0 || memcmp(want.data(), got.data(), isize) || (isize && rc != Z_STREAM_END)) ++bad;
            // a truncated stream must be refused, not over-read
            if (isize > 100 && brc::inflate::inflate_block(brc::inflate::Lanes{0, 1}, h + hdr, (total - hdr - 8) / 2, got.data(), isize, T) == 0) ++bad;
            ++nblk; o += total;
        }
    }
    printf("%d %d\n", nblk, bad);
    return bad != 0;
}
'''


def test_deflate_core_matches_zlib_on_every_block(tmp_path):
    """The exact DEFLATE code the kernel runs (host+device source), block by block against zlib: dynamic, fixed and stored blocks."""
    src = os.path.join(str(tmp_path), "h.cpp")
    open(src, "w").write(HARNESS)
    exe = os.path.join(str(tmp_path), "h")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "bam_readcount_b200", "csrc"), "-o", exe, src, "-lz"])
    files = [os.path.join(GOLDEN, "test.bam"), os.path.join(GOLDEN, "test_bad_rg.bam")]
    from bam_readcount_b200 import synth_cb
    sp = synth_cb.Spec(seed=2, contig_len=1280 * 200)
    for lv in (6, 0, 1):                               # default, stored blocks, fast compression
        d = tmp_path / f"level{lv}"
        d.mkdir()
        files.append(bamwrite.write_sample_bam(sp, 0, 0, 120, str(d), level=lv)["bam"])
    nblk, bad = map(int, subprocess.check_output([exe] + files).split())
    assert bad == 0 and nblk >= 20


def test_bai_span_covers_the_fetch():
    bai = bamio.BaiIndex(os.path.join(GOLDEN, "test.bam.bai"))
    sp = bamio.bam_span(os.path.join(GOLDEN, "test.bam"), bai, 20, 10402984, 10405200)
    assert sp is not None and sp["entries"] == sorted(sp["entries"]) and len(sp["comp"]) > 1000
    assert bamio.bam_span(os.path.join(GOLDEN, "test.bam"), bai, 3, 100, 200) is None
    w = bai.window_weights(20, 700)
    assert w.sum() > 0 and w[:600].sum() == 0               # all the coverage sits around 10.4 Mb


def _records_of(batch, idx):
    b = batch.select(idx)
    return [(int(b.pos[i]), int(b.flag[i]), int(b.mapq[i]), int(b.l_qseq[i]), int(b.nm[i]), int(b.sm[i]), int(b.lib[i]),
             b.cigar[int(b.cigar_off[i]):int(b.cigar_off[i + 1])].tobytes(), b.seq[int(b.seq_off[i]):int(b.seq_off[i + 1])].tobytes(),
             b.qual[int(b.qual_off[i]):int(b.qual_off[i + 1])].tobytes()) for i in range(b.n_reads)]


@pytest.mark.gpu
def test_device_decoded_batch_equals_host_decoder():
    from bam_readcount_b200.engine import Engine
    jobs = [(os.path.join(GOLDEN, "test.bam"), 20, 10402000, 10406000), (os.path.join(GOLDEN, "test_bad_rg.bam"), 20, 10402984, 10402985)]
    from bam_readcount_b200 import synth_cb
    sp = synth_cb.Spec(seed=6, contig_len=1280 * 2000)
    info = bamwrite.write_sample_bam(sp, 0, 0, 1500, tempfile.mkdtemp())
    jobs += [(info["bam"], 0, 200_000, 1_500_000), (info["bam"], 0, 0, 50_000)]
    e = Engine(per_lib=True, lib_names=["a"] * 16)
    try:
        for path, tid, beg, end in jobs:
            hdr, host = bamio.read_bam(path)
            rg_lib = {rg: hdr.lib_of_rg(rg) for rg in hdr.rg_lb}
            bai = bamio.BaiIndex(path + ".bai")
            span = bamio.bam_span(path, bai, tid, beg, end, rg_lib)
            dev = e.decode_bam_span(span)
            want = _records_of(host, host.fetch(tid, beg, end))
            got = _records_of(dev, np.arange(dev.n_reads))
            # the span holds every record samfetch yields, in file order (plus neighbours the kernels ignore)
            pos = {r: i for i, r in enumerate(got)}
            assert all(r in pos for r in want), path
            idx = [pos[r] for r in want]
            assert idx == sorted(idx)
            assert len(span["entries"]) >= 1 and dev.n_reads >= len(want)
    finally:
        e.close()


@pytest.mark.gpu
@pytest.mark.parametrize("flags", [dict(), dict(per_lib=True, insertion_centric=True, min_mapq=10, min_bq=15)])
def test_region_from_compressed_span_equals_region_from_host_reads(flags):
    """brc_push_bam_span (inflate + framing + kernels, reads never on the host) == brc_push_reads of the host-decoded records."""
    from bam_readcount_b200.engine import Engine
    from bam_readcount_b200 import synth_cb
    sp = synth_cb.Spec(seed=12, contig_len=1280 * 600)
    info = bamwrite.write_sample_bam(sp, 0, 0, 600, tempfile.mkdtemp())
    hdr, host = bamio.read_bam(info["bam"])
    libs = hdr.lib_names
    rg_lib = {rg: hdr.lib_of_rg(rg) for rg in hdr.rg_lb}
    ref = sp.ref_host(0, 0, info["length"])
    beg, end = 100_000, 700_000
    texts = []
    for mode in ("host", "span"):
        e = Engine(lib_names=libs, **flags)
        try:
            e.set_reference(0, "chr1", info["length"], ref, 0)
            e.begin_region(0, beg, end, False)
            if mode == "host":
                e.push_reads(host.select(host.fetch(0, beg - 1, end)))
            else:
                e.push_bam_span(bamio.bam_span(info["bam"], bamio.BaiIndex(info["bam"] + ".bai"), 0, beg - 1, end, rg_lib))
            e.end_region()
            e.compute()
            texts.append(e.format_text(-1))
        finally:
            e.close()
    assert texts[0] == texts[1] and len(texts[0].splitlines()) == end - beg


@pytest.mark.gpu
def test_cli_device_decode_matches_host_decode(tmp_path):
    """brc-readcount with BRC_CLI_DEVICE_DECODE=1 (compressed spans -> GPU inflate/framing) prints what the host-decode path prints."""
    from bam_readcount_b200 import build, synth_cb
    exe = build.build_cli()
    sp = synth_cb.Spec(seed=21, contig_len=1280 * 500)
    info = bamwrite.write_sample_bam(sp, 0, 0, 500, str(tmp_path))
    for extra in ([], ["-p", "-q", "20", "-b", "20"]):
        args = [exe, "-w", "0"] + extra + ["-f", info["fasta"], info["bam"], "chr1:5001-600000"]
        env = dict(os.environ, BRC_CLI_WINDOW="150000")
        host = subprocess.run(args, capture_output=True, env=env)
        dev = subprocess.run(args, capture_output=True, env=dict(env, BRC_CLI_DEVICE_DECODE="1"))
        assert host.returncode == 0 and dev.returncode == 0, dev.stderr.decode()[-1500:]
        assert dev.stdout == host.stdout and len(host.stdout.splitlines()) == 595000
