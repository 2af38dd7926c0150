"""Counter-based workload generator (include/brc_synth.h) and the streaming / sharding driver (bam_readcount_b200/stream.py).

CPU: the host generator is deterministic and window-independent, its distributions are the survey's, the SAM it writes is the
batch it returns (checked through the reference binary == oracle), shards partition the windows, and the ordered-emit transport
works between two gloo ranks.  GPU: the device generator is byte-identical to the host one, the packed records decode to the
full-width view, and a region computed window by window equals the region computed at once.
"""
import os
import socket

import numpy as np
import pytest

import cases
from bam_readcount_b200 import stream as st
from bam_readcount_b200 import synth_cb as sc

FIELDS = ("pos", "flag", "mapq", "lib", "l_qseq", "nm", "sm", "cigar_off", "cigar", "seq_off", "seq", "qual_off", "qual")


def _spec(**kw):
    return sc.Spec(seed=77, contig_len=1280 * 400, n_contigs=3, **kw)


def test_host_generator_is_deterministic_and_window_independent():
    sp = _spec()
    a, _ = sp.window_host(1, 10, 30, threads=4)
    b, _ = sp.window_host(1, 10, 30, threads=1)
    for f in FIELDS:
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    # the reads of a block do not depend on the window they are generated in
    c, _ = sp.window_host(1, 20, 25)
    lo, hi = 10 * 256, 15 * 256
    assert np.array_equal(a.pos[lo:hi], c.pos)
    assert np.array_equal(a.qual[lo * 150:hi * 150], c.qual)
    assert np.array_equal(a.seq[lo * 75:hi * 75], c.seq)
    assert np.array_equal(a.nm[lo:hi], c.nm)
    # another contig, another seed: different data
    d, _ = sp.window_host(2, 10, 30)
    assert not np.array_equal(a.qual, d.qual)
    assert np.all(np.diff(a.pos) >= 0) and a.pos.min() >= 10 * 1280 and a.pos.max() < 30 * 1280


def test_host_generator_distributions_match_the_survey():
    sp = sc.Spec(seed=1234, contig_len=1280 * 2000)
    b, _ = sp.window_host(0, 0, 800)
    n = b.n_reads
    assert n == 800 * 256
    ncig = np.diff(b.cigar_off.astype(np.int64))
    assert abs((ncig == 1).mean() - 0.90) < 0.01 and abs((ncig == 2).mean() - 0.04) < 0.005 and abs((ncig == 3).mean() - 0.06) < 0.006
    assert abs((b.flag == 16).mean() - 0.5) < 0.01
    mq = np.bincount(b.mapq, minlength=61) / n
    assert abs(mq[60] - 0.5) < 0.01 and abs(mq[40] - 1 / 6) < 0.01 and abs(mq[0] - 1 / 6) < 0.01
    q = b.qual.reshape(n, 150)
    assert set(np.unique(q)) <= {2, 12, 25, 30, 37}
    fwd = b.flag == 0
    tail = (q[:, -1] == 2)
    assert abs(tail[fwd].mean() - (0.2 + 0.8 / 7)) < 0.02          # 20 % Q2 tails + iid Q2 on the last base
    # substitutions: NM - indel bases ~ Binomial(150, 0.005)
    first_op_len = b.cigar[b.cigar_off[:-1].astype(np.int64)] >> 4
    indel = np.where(ncig == 3, np.where(first_op_len == 70, 2, 3), 0)
    subs = b.nm - indel
    assert subs.min() >= 0 and abs(subs.mean() - 0.75) < 0.02
    # reads agree with the reference except at substitutions
    ref = np.frombuffer(sp.ref_host(0, 0, 2000 * 1280), dtype=np.uint8)
    code = np.zeros(256, np.uint8); code[ord("A")] = 1; code[ord("C")] = 2; code[ord("G")] = 4; code[ord("T")] = 8
    simple = np.nonzero(ncig == 1)[0][:500]
    mism = 0
    for i in simple:
        s = b.seq[i * 75:(i + 1) * 75]
        nib = np.empty(150, np.uint8); nib[0::2] = s >> 4; nib[1::2] = s & 15
        mism += int((nib != code[ref[b.pos[i]:b.pos[i] + 150]]).sum()) - int(b.nm[i])
    assert mism == 0


def test_deep_mode_groups_reads_per_site():
    sp = sc.Spec(seed=5, mode=sc.DEEP, n_libs=8, depth=1000, site_stride=700, n_sites=6, contig_len=1280)
    b, ror = sp.window_host(0, 2, 5)
    assert b.n_reads == 3000 and np.array_equal(ror, np.repeat(np.arange(3), 1000))
    end = b.ref_end()
    for k in range(3):
        p = sp.site_pos(2 + k)
        sl = slice(k * 1000, (k + 1) * 1000)
        assert np.all(b.pos[sl] <= p) and np.all(end[sl] > p) and np.all(np.diff(b.pos[sl]) >= 0)
    assert np.all(np.diff(b.pos) >= 0)


SAMPLE = (sc.Spec(seed=1234, contig_len=1280 * 5000, n_contigs=2), 12, 1280 * 2, 1280 * 9)     # spec, blocks, region [beg, end)
SAMPLE_FLAGS = ((["-i"], dict(insertion_centric=True)), (["-q", "20", "-b", "20", "-p"], dict(min_mapq=20, min_bq=20, per_lib=True)))


def test_generated_bam_reference_binary_equals_oracle(tmp_path):
    """The SAM the generator writes is the batch it returns: byte for byte the SAM synth.write_sam makes of that batch, and the
    reference binary's STDOUT on it (through samtools; stored as digests in tests/golden/reference_outputs.json) equals the
    oracle on the batch."""
    import ctypes
    from bam_readcount_b200 import synth
    from oracle.oracle import Oracle
    sp, blocks, beg, end = SAMPLE
    length = min(blocks * 1280 + 400, sp.contig_len)                 # the @SQ length write_sample_bam declares
    b, _ = sp.window_host(0, 0, blocks)
    gen, want = tmp_path / "gen.sam", tmp_path / "want.sam"
    assert sc.load().brc_synth_write_sam(ctypes.byref(sp.c), 0, 0, blocks, str(gen).encode(), b"chr1", length, 4) == 0
    synth.write_sam(str(want), b, [("chr1", length)], n_libs=8)
    assert gen.read_bytes() == want.read_bytes()
    for argv, flags in SAMPLE_FLAGS:
        o = Oracle(lib_names=[f"lib{i}" for i in range(8)], **flags)
        o.region(b.select(b.fetch(0, beg - 1, end)), tid=0, beg=beg, end=end, contig="chr1", chrom_len=length,
                 ref_seq=sp.ref_host(0, 0, length), ref_win_beg=0, site_list_mode=False)
        cases.assert_reference_output("synth_sample " + " ".join(argv), o.text().encode("latin-1"))


def test_windows_and_weighted_shards_partition_the_genome():
    sp = sc.Spec(seed=1, contig_len=1280 * 1003, n_contigs=5)
    wins = st.wgs_windows(sp, 10)
    assert len(wins) == 50
    for c in range(5):
        cw = [w for w in wins if w.contig == c]
        assert cw[0].beg == 0 and cw[-1].end == sp.contig_len and all(cw[i].end == cw[i + 1].beg for i in range(9))
        assert all(w.blk_lo == max(w.beg // 1280 - 1, 0) and w.blk_hi * 1280 == w.end for w in cw)
    weights = [sp.window_reads(w.blk_lo, w.blk_hi) for w in wins]
    for world in (1, 2, 3, 4, 8, 64):
        sh = st.plan_shards_weighted(weights, world)
        assert sh[0][0] == 0 and sh[-1][1] == len(wins) and all(sh[i][1] == sh[i + 1][0] for i in range(world - 1))
        if world <= 8:
            tot = [sum(weights[a:b]) for a, b in sh]
            assert max(tot) - min(tot) <= 2.01 * max(weights)      # every cut is within half a unit of its target
    # skewed coverage: the heavy unit gets a shard of its own
    sh = st.plan_shards_weighted([1, 1, 1, 100, 1, 1], 3)
    assert any(a <= 3 < b and b - a <= 2 for a, b in sh)
    assert st.plan_shards_weighted([], 2) == [(0, 0), (0, 0)]


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close(); return p


def _gather_worker(rank, world, port, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    got = []
    ring = st.GatherRing(rank, world, torch.device("cpu"), 4096, 4096, consume=lambda src, tw, ts: got.append((src, tw.clone(), ts.clone())))
    rng = np.random.default_rng(rank)
    sent = []
    for k in range(3):                                   # three rounds; rank 1 has nothing in the last one (ragged shards)
        nw = 0 if (rank == 1 and k == 2) else 32 * (k + 1 + rank)
        ns = 72 * (k if rank == 1 else 0)
        tw = torch.from_numpy(rng.integers(0, 256, nw, dtype=np.uint8))
        ts = torch.from_numpy(rng.integers(0, 256, ns, dtype=np.uint8))
        sent.append((tw, ts))
        ring.round(tw, ts)
    # the size-exchange-free protocol (fixed message sizes known from the shard plan): words, pool bound, 4-byte count
    fixed_sent = []
    for k in range(5):                                   # five rounds: both spool sets of rank 0 are reused
        nw, ns = 64 * (k + 1), 144
        mine = None
        if rank == 1:
            mine = (torch.from_numpy(rng.integers(0, 256, nw, dtype=np.uint8)), torch.from_numpy(rng.integers(0, 256, ns, dtype=np.uint8)),
                    torch.from_numpy(np.array([k + 1], dtype=np.int32).view(np.uint8).copy()))
            fixed_sent.append((mine[0], mine[1]))
        ring.round_fixed(mine, {1: (nw, ns)} if rank == 0 else {})
    sent += fixed_sent
    q.put((rank, [(s, a.numpy().tobytes(), b.numpy().tobytes()) for s, a, b in got], [(a.numpy().tobytes(), b.numpy().tobytes()) for a, b in sent]))
    dist.barrier()
    dist.destroy_process_group()


def test_gather_ring_two_ranks_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict()
    for _ in range(2):
        r, got, sent = q.get(timeout=120)
        res[r] = (got, sent)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    got0, _ = res[0]
    _, sent1 = res[1]
    assert [g[0] for g in got0] == [1] * 8                 # three variable-size rounds + five fixed-size rounds
    assert [(g[1], g[2]) for g in got0] == sent1          # rank 0 received rank 1's records, round by round, byte for byte
    assert res[1][0] == []


# ------------------------------------------------------------------------------------------------ GPU
@pytest.mark.gpu
def test_device_generator_equals_host_generator():
    import torch
    dev = torch.device("cuda", 0)
    for sp, lo, hi in ((_spec(), 5, 45), (sc.Spec(seed=9, contig_len=1280 * 64), 60, 64),
                       (sc.Spec(seed=5, mode=sc.DEEP, n_libs=8, depth=1000, site_stride=700, n_sites=6, contig_len=1280), 1, 4)):
        dw = sc.DeviceWindow(sp, sp.window_reads(lo, hi) + 512, dev)
        dw.fill(1 if sp.mode == sc.WGS and sp.n_contigs > 1 else 0, lo, hi, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        d = dw.to_host()
        h, ror = sp.window_host(1 if sp.mode == sc.WGS and sp.n_contigs > 1 else 0, lo, hi)
        for f in FIELDS:
            assert np.array_equal(getattr(d, f), getattr(h, f)), f
        if sp.mode == sc.DEEP:
            assert np.array_equal(dw.t["region"][:d.n_reads].cpu().numpy(), ror)
        L = 5000
        ra = torch.empty(L, dtype=torch.uint8, device=dev)
        sc.load().brc_synth_ref_device(__import__("ctypes").byref(sp.c), 0, 123, L, ra.data_ptr(), torch.cuda.current_stream().cuda_stream)
        assert ra.cpu().numpy().tobytes() == sp.ref_host(0, 123, L)


@pytest.mark.gpu
def test_packed_records_decode_to_the_full_width_view():
    from bam_readcount_b200.engine import Engine
    for case, flags in ((cases.synthetic_case(L=20000, depth=40, seed=11, regions=((0, 1000, 19000),)), dict(per_lib=True)),
                        (cases.deep_case(n_sites=2, depth=3000, seed=3), dict()),           # depth > 255: every site escapes
                        (cases.deep_case(n_sites=2, depth=700, seed=4), dict(per_lib=True))):
        e = Engine(lib_names=case["lib_names"], **flags)
        try:
            for ci, (name, clen, seq, wb) in enumerate(case["contigs"]):
                e.set_reference(ci, name, clen, seq, wb)
            for (ci, b1, e1) in case["regions"]:
                tid, beg, end, sub = cases.region_reads(case, ci, b1, e1)
                e.begin_region(tid, beg, end, True)
                e.push_reads(sub)
                e.end_region()
            res = e.compute()
            pk = e.packed()
            ncover, npass, flg, pbase, ps = pk.widen()
            assert np.array_equal(ncover, res.ncover) and np.array_equal(npass, res.npass) and np.array_equal(flg, res.flags)
            assert np.array_equal(pbase, res.pbase) and np.array_equal(ps, res.pstats)
            assert pk.words.nbytes == 32 * res.n_rows * res.n_slots
            esc = int(((pk.words[1] & 7) == 7).sum())
            if "deep" in case["name"] and not flags:
                assert esc > 0
        finally:
            e.close()


@pytest.mark.gpu
def test_windowed_device_path_equals_whole_region():
    """A contig walked window by window on the device path (generator in HBM -> plan -> run, the bench's C4 loop) gives,
    site for site, the records of the same contig pushed as ONE region through the host path."""
    import torch
    from bam_readcount_b200.engine import Engine
    dev = torch.device("cuda", 0)
    sp = sc.Spec(seed=4321, contig_len=1280 * 120, n_contigs=2)
    flags = dict(insertion_centric=True)
    wins = [w for w in st.wgs_windows(sp, 5) if w.contig == 1]
    hb, _ = sp.window_host(1, 0, 120)
    ref = sp.ref_host(1, 0, sp.contig_len)
    e = Engine(**flags)
    e.set_reference(1, "chr2", sp.contig_len, ref, 0)
    e.begin_region(1, 0, sp.contig_len, False)
    e.push_reads(hb)
    e.end_region()
    whole = e.compute()
    wdump = whole.dump(hb, {1: (0, ref)})
    e.close()
    run = st.WindowRunner(sp, max(sp.window_reads(w.blk_lo, w.blk_hi) for w in wins), dev, flags)
    try:
        for w in wins:
            run.busy = False
            run.launch(w)
            torch.cuda.synchronize()
            r = run.eng.fetch_device_results(run.stream.cuda_stream)
            a, b = w.first_pos, w.end
            sub, _ = sp.window_host(1, w.blk_lo, w.blk_hi)
            got = r.dump_range(sub, {1: (0, ref)}, 0, a, b)
            want = whole.dump_range(hb, {1: (0, ref)}, 0, a, b)
            assert got == want
            s0 = w.beg - w.first_pos
            uncovered = w.n_sites - int((r.ncover[0, s0:] > 0).sum())          # only the first bases of a contig can lack a spanning read
            assert uncovered == 0 or (w.beg == 0 and uncovered < 64)
    finally:
        run.close()
    assert len(wdump) > 0


@pytest.mark.gpu
def test_site_at_50000x_eight_libraries_is_bit_exact():
    """BASELINE config 5's depth: one panel site under 50 000 reads, -p with 8 libraries, -d 100000000 — the depth at which the
    reference's own sequential-float drift exceeds 1e-6 (SURVEY.md Appendix D), so only the ordered sums match."""
    from bam_readcount_b200.engine import Engine
    from oracle.oracle import Oracle
    sp = sc.Spec(seed=1234, mode=sc.DEEP, n_libs=8, depth=50_000, site_stride=1000, n_sites=4, contig_len=1280)
    libs = [f"lib{i}" for i in range(8)]
    L = sp.deep_contig_len()
    ref = sp.ref_host(0, 0, L)
    hb, _ = sp.window_host(0, 1, 2)
    p = sp.site_pos(1)
    for flags in (dict(per_lib=True, max_cnt=100_000_000), dict(max_cnt=100_000_000)):
        o = Oracle(lib_names=libs, **flags)
        o.region(hb, tid=0, beg=p, end=p + 1, contig="chr1", chrom_len=L, ref_seq=ref, ref_win_beg=0, site_list_mode=True)
        e = Engine(lib_names=libs, **flags)
        try:
            e.set_reference(0, "chr1", L, ref, 0)
            e.begin_region(0, p, p + 1, True)
            e.push_reads(hb)
            e.end_region()
            res = e.compute()
            assert res.dump(hb, {0: (0, ref)}) == o.dump()
            assert e.format_text(-1) == o.text()
            assert int(res.ncover[:, 1].sum()) == 50_000
        finally:
            e.close()


@pytest.mark.gpu
def test_gather_checksum_is_a_function_of_the_bytes_only():
    """bench.py verifies the NCCL gather by comparing the senders' checksums with rank 0's: the value must not depend on the
    buffer's alignment, must match the documented formula (include/brc_synth.h) and must move when a byte or a length does."""
    import torch
    dev = torch.device("cuda", 0)
    rng = np.random.default_rng(11)

    def formula(b: bytes) -> int:
        w = np.frombuffer(b + b"\0" * (-len(b) % 16), dtype="<u8").reshape(-1, 2)
        lo, hi = w[:, 0], w[:, 1]
        rot = (hi << np.uint64(29)) | (hi >> np.uint64(35))
        g = np.arange(len(w), dtype=np.uint64)
        with np.errstate(over="ignore"):
            return int((((lo ^ rot) + np.uint64(1)) * (np.uint64(2) * g + np.uint64(1))).sum(dtype=np.uint64))

    def device(t) -> int:
        acc = torch.zeros(1, dtype=torch.int64, device=dev)
        sc.checksum_device(t, acc, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
        return int(acc.cpu().numpy().view(np.uint64)[0])

    for n in (4, 12, 16, 20, 4096, 1_000_004, 3_000_000):
        raw = rng.integers(0, 256, n, dtype=np.uint8)
        want = formula(raw.tobytes())
        base = torch.zeros(n + 64, dtype=torch.uint8, device=dev)
        for off in (0, 4, 8, 16):                                   # 16-byte aligned and not
            view = base[off:off + n]
            view.copy_(torch.from_numpy(raw))
            assert device(view) == want, (n, off)
        flipped = raw.copy(); flipped[n // 2] ^= 1
        view.copy_(torch.from_numpy(flipped))
        assert device(view) != want
        if n > 4:
            view.copy_(torch.from_numpy(raw))
            assert device(view[:n - 4]) != want
