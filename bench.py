#!/usr/bin/env python
"""bench.py — pileup positions/s of the B200 engine on the BASELINE.json workloads.

  --config c4 (default; the configuration the metric is quoted on): synthetic whole genome, 24 contigs x 125 Mb = 3.0 Gb, 30x,
      150 bp reads, --insertion-centric, ONE input split over N GPUs (strong scaling).  The genome is cut into 240 windows of
      12.5 Mb; windows are dealt to ranks as contiguous shards balanced by coverage weight; every rank walks its shard with
      three windows in flight (bam_readcount_b200/stream.py); the packed records of every window go to rank 0 over NCCL
      (ncclSend/ncclRecv) for the ordered emit.  A step = one pass over the whole genome.  3 Gb of decoded reads (165 GB) do
      not fit one GPU next to their results, so each window's reads are (re)generated in HBM by the counter-based generator
      (bam_readcount_b200/csrc/brc_synth.cu) right before its kernels run; the generator's own time is INSIDE the timed region
      and reported separately (`config.gen_ms_per_window`).
  --config c3: synthetic 10 Mb contig, 30x, -q 20 -b 20, one region, inputs resident in HBM (kernel roofline detail).
  --config c5: ultra-deep panel, 10 000 sites x 50 000x x 8 libraries, -p -d 100000000, sites split over N GPUs.

  value : whole-job positions/s, device-timed (CUDA events, max over ranks), inputs produced in / resident in HBM
  e2e   : positions/s through the C ABI with HOST buffers: brc_push_reads (pinned host batch) -> brc_compute -> packed
          records back in host memory, H2D and D2H inside the timed region
  --impl reference : the UNMODIFIED reference binary (oracle/_ref/bam-readcount) on a bounded sample of the same workload,
          one process per EFFECTIVE host core over disjoint slices.
After the timed steps (outside the timed region) every rank re-runs 3 of its windows and diffs a sampled range of each against
the CPU oracle on the host-generated copy of the same reads (`parity`).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "pileup positions/sec"
UNIT = "positions/s"
LIBS = [f"lib{i}" for i in range(8)]

CONFIGS = {
    "c4": dict(workload="C4: synthetic whole genome 24 x 124 999 680 bp = 3.0 Gb, 30x, 150 bp reads, --insertion-centric, "
                        "240 windows of 12.5 Mb sharded over the GPUs (strong scaling)",
               flags=dict(insertion_centric=True), argv=["-i"], n_contigs=24, contig_blocks=97656, windows_per_contig=10),
    "c3": dict(workload="C3: synthetic 10 Mb contig, 30x, 150 bp reads, -q 20 -b 20, one region, inputs resident in HBM (per GPU)",
               flags=dict(min_mapq=20, min_bq=20), argv=["-q", "20", "-b", "20"], n_contigs=1, contig_blocks=7812, windows_per_contig=1),
    "c5": dict(workload="C5: ultra-deep panel, 10 000 single-base sites x 50 000x, 8 libraries, -p -d 100000000, sites sharded over the GPUs",
               flags=dict(per_lib=True, max_cnt=100_000_000), argv=["-p", "-d", "100000000"], n_sites=10_000, depth=50_000, site_stride=1000,
               sites_per_window=296),
}


def make_spec(cfg_name, args):
    from bam_readcount_b200 import synth_cb
    c = CONFIGS[cfg_name]
    if cfg_name == "c5":
        return synth_cb.Spec(seed=1234, mode=synth_cb.DEEP, n_libs=8, depth=args.c5_depth, site_stride=c["site_stride"], n_sites=args.c5_sites,
                             contig_len=synth_cb.BLOCK_BP)
    nb = c["contig_blocks"] if not args.contig_blocks else args.contig_blocks
    return synth_cb.Spec(seed=1234, mode=synth_cb.WGS, n_libs=8, contig_len=nb * synth_cb.BLOCK_BP,
                         n_contigs=args.contigs or c["n_contigs"])


# ------------------------------------------------------------------------------------------------
# host cores: what the lease can really use
# ------------------------------------------------------------------------------------------------
def affinity_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def cgroup_cpu_limit():
    """CPU quota of this cgroup in cores (cgroup v2 cpu.max / v1 cfs quota), or None when unlimited / unreadable."""
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            return float(q) / float(p)
    except Exception:
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0:
            return q / p
    except Exception:
        pass
    return None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def profiled_traffic():
    """DRAM bytes per K1 launch from the newest committed `ncu --set full` capture (profiles/traffic_*.json): a PROFILE
    constant of the same kernel on the C3 window, not measured in this run."""
    import glob
    fs = sorted(glob.glob(os.path.join(ROOT, "profiles", "traffic_*.json")))
    if not fs:
        return None, None
    try:
        d = json.load(open(fs[-1]))
        return float(d["pileup_kernel"]["traffic"]), os.path.basename(fs[-1]) + " (ncu capture of the C3 window; not measured in this run)"
    except Exception:
        return None, None


# ------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference binary on a bounded sample, N processes over DISJOINT slices
# ------------------------------------------------------------------------------------------------
def _run_procs(cmds):
    """Run the commands concurrently, count output lines, return (lines, seconds)."""
    t0 = time.perf_counter()
    ps = [subprocess.Popen(c, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL) for c in cmds]
    outs = []

    def drain(p):
        n = 0
        for chunk in iter(lambda: p.stdout.read(1 << 20), b""):
            n += chunk.count(b"\n")
        outs.append(n)
    ths = [threading.Thread(target=drain, args=(p,)) for p in ps]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    for p in ps:
        p.wait()
    return sum(outs), time.perf_counter() - t0


class ReferenceSample:
    """A bounded sample of the workload as ref.fa + s.bam, and the reference command line per slice."""

    def __init__(self, cfg_name, spec, slices, slice_sites):
        from bam_readcount_b200 import synth_cb
        from oracle.oracle import REF_BIN, REF_SAMTOOLS
        self.cfg_name, self.spec, self.slices, self.slice_sites = cfg_name, spec, slices, slice_sites
        self.wd = tempfile.mkdtemp(prefix="brc_ref_")
        self.bin = REF_BIN
        self.argv = CONFIGS[cfg_name]["argv"]
        if cfg_name == "c5":
            self.info = synth_cb.write_sample_bam(spec, 0, 0, slices * slice_sites, self.wd, REF_SAMTOOLS)
            self.lists = []
            for p in range(slices):
                path = os.path.join(self.wd, f"sites{p}.txt")
                with open(path, "w") as fh:
                    for k in range(p * slice_sites, (p + 1) * slice_sites):
                        fh.write(f"chr1\t{spec.site_pos(k) + 1}\t{spec.site_pos(k) + 1}\n")
                self.lists.append(path)
        else:
            nblk = -(-(slices * slice_sites) // synth_cb.BLOCK_BP) + 1
            self.info = synth_cb.write_sample_bam(spec, 0, 0, nblk, self.wd, REF_SAMTOOLS)

    def cmd(self, p, sites=None):
        base = [self.bin, "-w", "0"] + self.argv + ["-f", self.info["fasta"]]
        if self.cfg_name == "c5":
            return base + ["-l", self.lists[p], self.info["bam"]]
        n = self.slice_sites if sites is None else min(sites, self.slice_sites)
        b = p * self.slice_sites
        return base + [self.info["bam"], f"chr1:{b + 1}-{b + n}"]

    def step(self, procs, sites=None):
        return _run_procs([self.cmd(p, sites) for p in range(procs)])

    def close(self):
        shutil.rmtree(self.wd, ignore_errors=True)


def reference_measure(cfg_name, args, steps, warmup, size_steps=None):
    """1-process rate, effective parallelism, then `steps` timed steps with N = effective cores over disjoint slices."""
    from oracle.oracle import have_reference_binary
    if not have_reference_binary():
        return None
    spec = make_spec(cfg_name, args)
    aff = affinity_cores()
    quota = cgroup_cpu_limit()
    cap = int(min(aff, quota)) if quota else aff
    if cfg_name == "c5":
        slice_sites = args.ref_sample or 1          # one 50 000x site is ~0.5 s of reference time
        slices = min(cap, 8)
    else:
        slice_sites = args.ref_sample or max(5_000, min(150_000, 720_000 // max(size_steps or steps, 1)))
        slices = cap
    rs = ReferenceSample(cfg_name, spec, slices, slice_sites)
    try:
        cal = None if cfg_name == "c5" else min(slice_sites, 20_000)
        rs.step(1, cal)                                        # page the files in
        s1, t1 = rs.step(1, cal)
        r1 = s1 / t1
        sa, ta = rs.step(slices, cal)
        r_all = sa / ta
        # processes to run: the cgroup CPU quota when there is one (the lease's real core count), else the measured speed-up of
        # `slices` concurrent processes over one
        eff = int(max(1, min(slices, int(quota)))) if quota else int(max(1, min(slices, round(r_all / r1))))
        for _ in range(warmup):
            rs.step(eff, cal)
        tot_s, tot_t = 0, 0.0
        for _ in range(steps):
            s, dt = rs.step(eff)
            tot_s += s
            tot_t += dt
    finally:
        rs.close()
    value = tot_s / tot_t
    unit_s = "sites" if cfg_name == "c5" else "bp"
    sample = (f"{eff} concurrent reference processes over DISJOINT slices of {slice_sites} {unit_s} each of the same synthetic workload "
              f"(counter-based generator, seed 1234), stdout discarded; 1-process rate {r1:.0f} positions/s; {slices} processes "
              f"({aff} affinity cores, cgroup quota {quota}) reached {r_all:.0f} positions/s = {r_all / r1:.1f}x one process")
    return dict(value=value, ms_per_step=1000.0 * tot_t / max(steps, 1), eff=eff, r1=r1, r_all=r_all, slices=slices, slice_sites=slice_sites,
                affinity=aff, quota=quota, sample=sample)


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    m = reference_measure(args.config, args, args.steps, min(args.warmup, 1), size_steps=max(args.steps, 20))
    if m is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/bam-readcount not built (run oracle/build_ref.sh where /root/reference exists)"}))
        return 0
    line = {
        "impl": "reference", "metric": METRIC, "value": m["value"], "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": m["ms_per_step"], "higher_is_better": True,
        "scaling": "weak" if args.config == "c3" else "strong", "vs_baseline": None, "dtype": "u32+f32", "data": "synthetic",
        "config": {"workload": CONFIGS[args.config]["workload"], "sample_per_process": m["slice_sites"], "processes": m["eff"],
                   "one_process_positions_per_s": m["r1"], "effective_cores": m["eff"], "affinity_cores": m["affinity"], "cgroup_quota": m["quota"]},
        "cpu_baseline": {"value": m["value"], "unit": UNIT, "cores": m["eff"], "kind": "reference", "sample": m["sample"]},
        "e2e": {"value": m["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int):
        self.index = index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}",
                 "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                 "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for k, nm in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa(local: int):
    """Pin this rank's threads (and so its first-touch pinned allocations) to the NUMA node its GPU hangs off
    (SCALE_r01.json: GPU0-3 on node 0, GPU4-7 on node 1; unbound ranks made 8-GPU e2e 0.56 efficient)."""
    try:
        bus = subprocess.check_output(["nvidia-smi", f"--id={local}", "--query-gpu=pci.bus_id", "--format=csv,noheader"], text=True).strip().lower()
        if len(bus.split(":")[0]) == 8:      # 00000000:1b:00.0 -> 0000:1b:00.0
            bus = bus[4:]
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read())
        if node < 0:
            return {"numa_node": node}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus += list(range(int(lo), int(hi or lo) + 1))
        allowed = set(os.sched_getaffinity(0)) & set(cpus)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception as ex:   # binding is an optimisation, never fatal
        return {"error": str(ex)[:100]}


def batch_nbytes(b) -> int:
    return int(sum(getattr(b, k).nbytes for k in ("pos", "flag", "mapq", "lib", "l_qseq", "nm", "sm", "cigar_off", "cigar", "seq_off", "seq",
                                                  "qual_off", "qual")))


def oracle_dump(spec, flags, contig, pos_lo, pos_hi, lib_names):
    """CPU oracle on the host-generated reads around [pos_lo, pos_hi): region (pos_lo+1, pos_hi), halo pos_lo.
    Returns (dump text, host sub-batch, its first block)."""
    from bam_readcount_b200 import synth_cb
    from oracle.oracle import Oracle
    blo = max(pos_lo // synth_cb.BLOCK_BP - 1, 0)
    bhi = min(-(-pos_hi // synth_cb.BLOCK_BP), spec.blocks_per_contig())
    hb, _ = spec.window_host(contig, blo, bhi)
    beg, end = pos_lo + 1, pos_hi
    ref_end = min(spec.contig_len, bhi * synth_cb.BLOCK_BP + 400)
    ref = spec.ref_host(contig, 0, ref_end) if ref_end < 50_000_000 else None
    wb = 0
    if ref is None:
        wb = max(blo * synth_cb.BLOCK_BP - 400, 0)
        ref = spec.ref_host(contig, wb, ref_end - wb)
    o = Oracle(lib_names=lib_names, **flags)
    sub = hb.select(hb.fetch(contig, beg - 1, end))
    o.region(sub, tid=contig, beg=beg, end=end, contig=f"chr{contig + 1}", chrom_len=spec.contig_len, ref_seq=ref, ref_win_beg=wb,
             site_list_mode=False)
    return o.dump(), hb, blo, (wb, ref)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, handles):
    """--dump-outputs: the results the last timed step left in the engine handles (each handle's last window or launch), as a
    caller of brc_fetch_device_results receives them, on a fixed seeded sample of their sites, as DIR/<name>.npy (float64;
    the float32 statistics widened exactly).  Per sampled site: site_contig, site_pos (0-based), and per row ncover, npass,
    pbase, flags and the 13 statistics (stats); sec_records: the secondary records (indel alleles, further base classes) of
    the sampled sites, one per line as (site index, row, kind, indel length, read, qpos, 13 statistics), sorted."""
    from bam_readcount_b200.engine import N_STATS, _FLOAT_STATS
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(1234)

    def wide(st):
        out = st.astype(np.float64)
        for k in _FLOAT_STATS:
            out[k] = st[k].view(np.float32)
        return out

    cols = {k: [] for k in ("site_contig", "site_pos", "ncover", "npass", "pbase", "flags", "stats")}
    sec, n_done = [], 0
    for eng, stream in handles:
        res = eng.fetch_device_results(stream.cuda_stream)
        per_site = res.n_rows * (4 + N_STATS) * 8
        k = min(res.n_slots, DUMP_BYTES // 2 // len(handles) // per_site)
        pick = np.sort(rng.choice(res.n_slots, k, replace=False))
        contig, pos = np.zeros(res.n_slots), np.zeros(res.n_slots)
        for g in res.regions:
            contig[g["slot_base"]:g["slot_base"] + g["n_slots"]] = g["tid"]
            pos[g["slot_base"]:g["slot_base"] + g["n_slots"]] = g["first_pos"] + np.arange(g["n_slots"])
        cols["site_contig"].append(contig[pick])
        cols["site_pos"].append(pos[pick])
        for name in ("ncover", "npass", "pbase", "flags"):
            cols[name].append(getattr(res, name)[:, pick].T.astype(np.float64))
        cols["stats"].append(wide(res.pstats[:, :, pick]).transpose(2, 1, 0))
        for i, slot in enumerate(pick.tolist()):
            for row in range(res.n_rows):
                j = int(res.sec_head[row, slot])
                while j >= 0:          # the site's chain; the pool's order depends on the device's scheduling, hence the sort below
                    sec.append(np.concatenate([[n_done + i, row, res.sec_kind[j], res.sec_len[j], res.sec_read[j], res.sec_qpos[j]],
                                               wide(res.sec_stats[:, j])]))
                    j = int(res.sec_next[j])
        n_done += k
    out = {name: np.concatenate(v) for name, v in cols.items()}
    sec = np.array(sec, dtype=np.float64).reshape(-1, 6 + N_STATS)
    sec = sec[np.lexsort(sec.T[::-1])]
    room = (DUMP_BYTES - sum(a.nbytes for a in out.values())) // sec[0].nbytes if len(sec) else 0
    out["sec_records"] = sec[:room]
    for name, a in out.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_wgs(args, cfg_name):
    import torch
    import torch.distributed as dist
    from bam_readcount_b200 import stream as st
    from bam_readcount_b200 import synth_cb
    from bam_readcount_b200.engine import Engine, N_WORDS, SEC_RECORD_BYTES, pin_batch

    cfg = CONFIGS[cfg_name]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU path")
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    numa = bind_to_gpu_numa(local)
    if world > 1:
        # the gather's send/recv kernels run on NCCL's own stream: make it a HIGH-PRIORITY stream, so that its CTAs are placed as
        # soon as a pileup launch drains instead of queueing behind the next window's persistent grid
        try:
            opts = dist.ProcessGroupNCCL.Options()
            opts.is_high_priority_stream = True
            dist.init_process_group("nccl", device_id=device, pg_options=opts)
        except Exception:
            dist.init_process_group("nccl", device_id=device)
        if args.reserve_ctas > 0:
            os.environ.setdefault("BRC_K1_RESERVE_CTAS", str(args.reserve_ctas))
    spec = make_spec(cfg_name, args)
    flags = cfg["flags"]
    resident = cfg_name == "c3"
    wpc = cfg["windows_per_contig"]
    if resident:
        # weak scaling: every rank owns one 10 Mb contig of its own (contig index = rank)
        spec.n_contigs = world
        all_windows = st.wgs_windows(spec, wpc)
        my_windows = [w for w in all_windows if w.contig == rank]
        shards = [(r, r + 1) for r in range(world)]
    else:
        all_windows = st.wgs_windows(spec, wpc)
        weights = [spec.window_reads(w.blk_lo, w.blk_hi) for w in all_windows]     # coverage weight (a BAM: BAI linear-index byte deltas)
        shards = st.plan_shards_weighted(weights, world)
        my_windows = all_windows[shards[rank][0]:shards[rank][1]]
    rounds = max(b - a for a, b in shards)
    max_reads = max(spec.window_reads(w.blk_lo, w.blk_hi) for w in all_windows)
    max_slots = max(w.n_slots for w in all_windows)
    n_runners = 1 if resident else 3
    runners = [st.WindowRunner(spec, max_reads, device, flags) for _ in range(n_runners)]
    comm = torch.cuda.Stream(device=device)
    acc = torch.zeros(max(world, 1) * 2, dtype=torch.int64, device=device)      # [src] received checksum, [world + src] sender-side checksum

    def consume(src, tw, ts):      # rank 0's emitter stand-in: read every received byte
        sp = torch.cuda.current_stream().cuda_stream
        if tw.numel():
            synth_cb.checksum_device(tw, acc[src:src + 1], sp)
        if ts.numel():
            synth_cb.checksum_device(ts, acc[src:src + 1], sp)

    # ---- residency: keep as many of the shard's windows in HBM as fit (the whole shard for N >= 2); the rest are regenerated in
    # the timed loop by the counter-based generator ----
    resident_dw = {}
    if not resident and not args.no_resident:
        free_b, _ = torch.cuda.mem_get_info(device)
        per_read = synth_cb.DeviceWindow.bytes_per_read()
        budget = free_b - int(args.hbm_margin_gb * (1 << 30)) - (st.GatherRing.spool_bytes(world, max_slots * 4 * N_WORDS, (max_slots // 3 + 8192) * SEC_RECORD_BYTES) if rank == 0 else 0)
        shared_scratch = torch.empty(max_reads // synth_cb.BLOCK_READS + 4, dtype=torch.int64, device=device)
        for wi, w in enumerate(my_windows):
            nr = spec.window_reads(w.blk_lo, w.blk_hi)
            need = nr * per_read + (1 << 20)
            if budget < need:
                break
            dwr = synth_cb.DeviceWindow(spec, nr, device, scratch=shared_scratch, with_region=False)
            dwr.fill(w.contig, w.blk_lo, w.blk_hi, torch.cuda.current_stream().cuda_stream)
            resident_dw[wi] = dwr
            budget -= need
        torch.cuda.synchronize()

    ring = st.GatherRing(rank, world, device, max_slots * 4 * N_WORDS, (max_slots // 3 + 8192) * SEC_RECORD_BYTES, consume=consume) if world > 1 else None

    # records per pool message: a fixed bound from the window's geometry (25 % above what this workload needs), so that a round
    # needs no size exchange and no host synchronisation; the true count travels with it and is checked after the pass
    def sec_msg_records(w):
        return int(w.n_slots * args.sec_msg_per_site) + 4096

    def gather_round(j, verify):
        run = runners[j % n_runners] if j < len(my_windows) else None
        with torch.cuda.stream(comm):
            mine = None
            if run is not None:
                comm.wait_event(run.done)                 # stream order only: the host does not wait for the window
                mine = run.packed_tensors_fixed(sec_msg_records(my_windows[j]))
                if verify and rank > 0:
                    sp = comm.cuda_stream
                    synth_cb.checksum_device(mine[0], acc[world + rank:world + rank + 1], sp)
                    synth_cb.checksum_device(mine[1], acc[world + rank:world + rank + 1], sp)
            peers = {}
            if rank == 0:
                for src in range(1, world):
                    a0, b0 = shards[src]
                    if resident:
                        a0, b0 = src, src + 1
                    if a0 + j < b0:
                        wj = all_windows[a0 + j]
                        rsj = wj.n_slots * (len(LIBS) if flags.get("per_lib") else 1)
                        peers[src] = (rsj * 4 * N_WORDS, min(sec_msg_records(wj), rsj // 4 + 4096) * SEC_RECORD_BYTES)
            ring.round_fixed(mine, peers)
            if run is not None:
                run.sent.record(comm)

    def one_pass(verify=False):
        lag = 0            # the gather of window k is queued right behind its kernels (stream order; no host wait)
        for k in range(rounds + (lag if world > 1 else 0)):
            if k < len(my_windows):
                if resident and runners[0].window is not None:
                    r0 = runners[0]
                    r0.stream.wait_event(r0.sent)                                           # the previous step's records have left the handle
                    r0.eng.run_device(r0.dw.c_batch(), None, r0.stream.cuda_stream)       # inputs stay resident: kernels only
                    with torch.cuda.stream(r0.stream):
                        r0.done.record(r0.stream)
                else:
                    runners[k % n_runners].launch(my_windows[k], resident=resident_dw.get(k))
            if world > 1 and k >= lag and k - lag < rounds:
                gather_round(k - lag, verify)

    def join_streams():
        cur = torch.cuda.current_stream()
        for r in runners:
            cur.wait_stream(r.stream)
        cur.wait_stream(comm)
        if ring is not None:
            ring.join(cur)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up (the first pass also verifies the gather: received checksum == sender's checksum) ----
    gather_ok = None
    for it in range(args.warmup):
        one_pass(verify=(it == 0))
        join_streams()
        torch.cuda.synchronize()
        if it == 0 and world > 1:
            dist.all_reduce(acc[world:], op=dist.ReduceOp.SUM)
            a = acc.cpu().tolist()
            gather_ok = all(a[s] == a[world + s] for s in range(1, world)) if rank == 0 else None
            acc.zero_()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        one_pass()
    join_streams()
    ev1.record()
    barrier()
    elapsed_ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, [(r.eng, r.stream) for r in sorted((r for r in runners if r.window is not None),
                                                                            key=lambda r: (r.window.contig, r.window.beg))])
    gather_overflow = 0
    if world > 1:
        for r_ in runners:
            if r_.window is not None and r_.n_sec_host is not None and int(r_.n_sec_host[0]) > sec_msg_records(r_.window):
                gather_overflow += 1
    # one more pass WITHOUT the gather (untimed for `value`): what the ordered emit costs the step
    nogather_ms = None
    if world > 1:
        saved_world = world
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        c0.record()
        world = 1
        try:
            one_pass()
        finally:
            world = saved_world
        join_streams()
        c1.record()
        barrier()
        nogather_ms = c0.elapsed_time(c1)
    # link probe (untimed): the same send/recv group with idle SMs — what rank 0's NVLink ingress takes when nothing else runs
    ingress_gbps = None
    if world > 1:
        nprobe = min(w.n_slots for w in all_windows) * 4 * N_WORDS * (len(LIBS) if flags.get("per_lib") else 1)
        reps = 8
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        src_words = st.alias_device_bytes(runners[0].eng.device_packed().words, nprobe, device) if rank > 0 else None
        barrier()
        with torch.cuda.stream(comm):
            for rep in range(reps + 1):
                if rep == 1:
                    p0.record(comm)
                if rank == 0:
                    ops = [dist.P2POp(dist.irecv, ring.spool_w[src][0][:nprobe], src) for src in range(1, world)]
                else:
                    ops = [dist.P2POp(dist.isend, src_words, 0)]
                for req in dist.batch_isend_irecv(ops):
                    req.wait()
            p1.record(comm)
        torch.cuda.synchronize()
        barrier()
        ingress_gbps = nprobe * (world - 1) * reps / (p0.elapsed_time(p1) / 1000.0) / 1e9
    n_my_sites = sum(w.n_sites for w in my_windows)
    per_window_launches = 3 + runners[0].eng.launch_count()     # generator (count, scan, fill) + engine kernels
    launches = len(my_windows) * args.steps * (runners[0].eng.launch_count() if resident else per_window_launches)

    # ---- untimed: generator alone, per-kernel times and algorithmic bytes on a resident window ----
    r0 = runners[0]
    w0 = my_windows[len(my_windows) // 2]
    torch.cuda.synchronize()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(r0.stream):
        g0.record(r0.stream)
        for _ in range(3):
            r0.dw.fill(w0.contig, w0.blk_lo, w0.blk_hi, r0.stream.cuda_stream)
        g1.record(r0.stream)
    torch.cuda.synchronize()
    gen_ms = g0.elapsed_time(g1) / 3
    r0.busy = False
    r0.launch(w0)
    torch.cuda.synchronize()
    k0s, k1s, steps_ms = [], [], []
    for _ in range(5):
        r0.eng.run_device(r0.dw.c_batch(), None, r0.stream.cuda_stream)
        k0s.append(r0.eng.stage_ms(0)); k1s.append(r0.eng.stage_ms(1)); steps_ms.append(r0.eng.stage_ms(2))
    res = r0.eng.fetch_device_results(r0.stream.cuda_stream)
    pk = r0.eng.packed()
    lo_s = w0.beg - w0.first_pos
    w_sites = int((res.ncover[:, lo_s:].sum(axis=0) > 0).sum())
    w_events = int(res.ncover[:, lo_s:].sum())
    w_keys = int((res.pstats[0] > 0).sum()) + int((res.sec_kind < 8).sum() if res.n_sec else 0)
    n_reads_w = r0.dw.n_reads
    n_cig_w = int(r0.dw.t["cigar_off"][n_reads_w].item())
    # ALGORITHMIC bytes of one window (SURVEY.md §8d): reads + reference + 16 B/site + 52 B/key
    alg_bytes = 16 * n_reads_w + 4 * n_cig_w + 75 * n_reads_w + 150 * n_reads_w + w0.n_slots + 16 * w_sites + 52 * w_keys
    packed_bytes = pk.nbytes()
    uncovered = w0.n_sites - w_sites

    # ---- untimed: parity of 3 sampled windows per rank against the CPU oracle ----
    parity = {"checked": False}
    if not args.no_parity:
        picks = sorted(set([0, len(my_windows) // 2, len(my_windows) - 1]))
        span = args.parity_sites
        checked, ok = [], True
        rng = np.random.default_rng(1000 + rank)
        for wi in picks:
            w = my_windows[wi]
            r0.busy = False
            r0.launch(w)
            torch.cuda.synchronize()
            rr = r0.eng.fetch_device_results(r0.stream.cuda_stream)
            a = int(rng.integers(w.first_pos, max(w.first_pos + 1, w.end - span)))
            b = min(a + span, w.end)
            od, hb, blo, (wb, ref) = oracle_dump(spec, flags, w.contig, a, b, [])
            ed = rr.dump_range(hb, {w.contig: (wb, ref)}, 0, a, b, read_offset=(blo - w.blk_lo) * synth_cb.BLOCK_READS)
            same = od == ed
            ok = ok and same
            checked.append({"window": shards[rank][0] + wi if not resident else rank, "contig": w.contig, "sites": [a, b], "identical": same,
                            "dump_bytes": len(od)})
        parity = {"checked": True, "identical": ok, "windows": checked, "what": "raw accumulator dump (integer and float bits) of a sampled "
                  f"{span}-site range per window vs oracle/brc_oracle.c on the host-generated copy of the same reads"}

    # ---- e2e: host buffers through the push path (admission scan + H2D + kernels + D2H of the packed records) ----
    e2e = None
    if args.e2e_windows > 0:
        import threading
        ne = min(args.e2e_windows, len(my_windows))
        # The caller keeps `nh` engine handles in flight, one host thread each (brc_compute blocks until the window's records are in
        # host memory): window k+1's upload runs under window k's result download, so both PCIe directions stay busy.
        nh = max(1, min(args.e2e_handles, ne))
        pool_n = min(max(2, nh), ne)
        engs = [Engine(device=local, **flags) for _ in range(nh)]
        hosts = []
        for w in my_windows[:pool_n]:
            hb, _ = spec.window_host(w.contig, w.blk_lo, w.blk_hi)
            hosts.append((w, pin_batch(hb), batch_nbytes(hb)))
        for c in sorted(set(w.contig for w, _, _ in hosts)):
            lo_p = max(min(w.blk_lo for w, _, _ in hosts if w.contig == c) * synth_cb.BLOCK_BP - 400, 0)
            hi_p = min(spec.contig_len, max(w.end for w, _, _ in hosts if w.contig == c) + 400)
            for en in engs:
                en.set_reference(c, f"chr{c + 1}", spec.contig_len, spec.ref_host(c, lo_p, hi_p - lo_p), lo_p)
        h2d = d2h = 0
        sites = 0
        times = []
        for it in range(args.e2e_steps + 1):
            tally = [[0, 0, 0, None] for _ in range(nh)]

            def handle_loop(i, first_pass=(it == 0)):
                en, tl = engs[i], tally[i]
                try:
                    for k in range(i, ne, nh):
                        w, hb, nb = hosts[k % pool_n]
                        en.reset()
                        en.begin_region(w.contig, w.beg, w.end, False)
                        en.push_reads(hb)
                        en.end_region()
                        en._check(en.lib.brc_compute(en.h))
                        tl[0] += en.h2d_bytes()      # what crossed PCIe (regular offsets / constant columns are rebuilt on the device)
                        tl[1] += w.n_sites
                        if first_pass:
                            tl[2] += en.packed().nbytes()
                except Exception as ex:          # surfaced after the join
                    tl[3] = ex

            barrier()
            t0 = time.perf_counter()
            if nh == 1:
                handle_loop(0)
            else:
                ths = [threading.Thread(target=handle_loop, args=(i,)) for i in range(nh)]
                for th in ths:
                    th.start()
                for th in ths:
                    th.join()
            dt = time.perf_counter() - t0
            for tl in tally:
                if tl[3] is not None:
                    raise tl[3]
            if it == 0:
                d2h_per = sum(tl[2] for tl in tally)
            else:
                times.append(dt)
            h2d, sites = sum(tl[0] for tl in tally), sum(tl[1] for tl in tally)
        for en in engs:
            en.close()
        e2e = dict(ms=1000.0 * sum(times) / len(times), sites=sites, h2d=h2d, d2h=d2h_per, windows=ne, handles=nh)

    # ---- reduce over ranks: max time, sum of units ----
    t = torch.tensor([elapsed_ms, e2e["ms"] if e2e else 0.0, nogather_ms or 0.0], device=device, dtype=torch.float64)
    u = torch.tensor([n_my_sites, e2e["sites"] if e2e else 0, e2e["h2d"] if e2e else 0, e2e["d2h"] if e2e else 0, launches,
                      1 if parity.get("identical", True) else 0], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        red = u.clone()
        dist.all_reduce(red, op=dist.ReduceOp.SUM)
        mn = u.clone()
        dist.all_reduce(mn, op=dist.ReduceOp.MIN)
        u = red
        parity_all = bool(mn[5].item() >= 1)
    else:
        parity_all = bool(parity.get("identical", True))
    elapsed_ms, e2e_max = float(t[0]), float(t[1])
    tot_sites = float(u[0])

    if rank == 0:
        ms_per_step = elapsed_ms / args.steps
        value = tot_sites / (ms_per_step / 1000.0)
        peak, peak_src = measured_peak_gbs()
        k1 = sum(k1s) / len(k1s)
        k0 = sum(k0s) / len(k0s)
        stp = sum(steps_ms) / len(steps_ms)
        ach = alg_bytes / (k1 / 1000.0) / 1e9
        traffic, traffic_src = profiled_traffic()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak" if resident else "strong", "vs_baseline": None,
            "dtype": "u32+f32 (f64 for one add)", "data": "synthetic",
            "config": {"workload": cfg["workload"], "flags": " ".join(cfg["argv"]), "genome_bp": spec.contig_len * spec.n_contigs,
                       "windows": len(all_windows), "windows_rank0": len(my_windows), "shards": shards,
                       "positions_per_step": tot_sites, "events_per_s": value * (w_events / max(w_sites, 1)),
                       "inputs": ("resident in HBM" if resident else
                                  f"{len(resident_dw)} of rank 0's {len(my_windows)} windows resident in HBM before the timed region; the others are "
                                  "(re)generated in HBM by the counter-based generator inside it"),
                       "windows_resident_rank0": len(resident_dw),
                       "gen_ms_per_window": gen_ms, "window_reads": n_reads_w, "window_sites": w_sites, "window_uncovered_sites": uncovered,
                       "window_events": w_events, "window_keys": w_keys, "window_packed_result_bytes": packed_bytes,
                       "l2": "every window's inputs (%.0f MB) exceed the 126 MB L2; no flush" % (alg_bytes / 1e6),
                       "gather": (None if world == 1 else {"transport": "NCCL send/recv of the packed records to rank 0, one group per round",
                                                           "k1_reserved_cta_slots": int(os.environ.get("BRC_K1_RESERVE_CTAS", "0")),
                                                           "rounds_per_step": rounds, "bytes_to_rank0_per_step": ring.bytes_received / max(args.steps + args.warmup, 1),
                                                           "verified_checksums": gather_ok, "rank0_ingress_probe_GBps": ingress_gbps, "pool_message_records_per_site": args.sec_msg_per_site,
                                                           "pool_message_overflows_rank0": gather_overflow,
                                                           "ms_per_step_without_gather": float(t[2]),
                                                           "positions_per_s_without_gather": tot_sites / (float(t[2]) / 1000.0) if float(t[2]) > 0 else None}),
                       "numa": numa},
            "roofline": {"bound": "hbm", "kernel": "pileup_kernel (K1), one window", "achieved": ach, "peak": peak, "unit": "GB/s",
                         "frac": ach / peak, "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": alg_bytes, "k1_ms": k1, "k0_ms": k0, "window_step_ms": stp,
                         "step_frac": alg_bytes / (stp / 1000.0) / 1e9 / peak},
            "gpu_launches": int(u[4]),
            "parity": dict(parity, all_ranks_identical=parity_all),
            "clocks": clocks,
        }
        if e2e:
            line["e2e"] = {"value": float(u[1]) / (e2e_max / 1000.0), "unit": UNIT, "h2d_bytes_per_step": int(u[2]), "d2h_bytes_per_step": int(u[3]),
                           "ms_per_step": e2e_max, "windows_per_rank": e2e["windows"], "handles_in_flight": e2e["handles"],
                           "what": "brc_push_reads(pinned host window) + brc_compute per window, the caller alternating between "
                                   f"{e2e['handles']} engine handle(s); results = packed records in pinned host memory"}
        if world == 1 and not args.no_cpu_baseline:
            try:
                m = reference_measure(cfg_name, args, 1, 0, size_steps=max(args.steps, 20))
                if m:
                    line["cpu_baseline"] = {"value": m["value"], "unit": UNIT, "cores": m["eff"], "kind": "reference", "sample": m["sample"],
                                            "one_process": m["r1"]}
            except Exception as ex:  # the baseline is a reported extra, never fatal for the GPU number
                line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "reference", "sample": f"failed: {ex}"}
        if world == 1 and not args.no_e2e_text:
            try:
                line["e2e_text"] = e2e_text(cfg_name, spec, args)
            except Exception as ex:
                line["e2e_text"] = {"value": None, "error": str(ex)[:200]}
        print(json.dumps(line))
    for r in runners:
        r.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def e2e_text(cfg_name, spec, args):
    """The whole pipeline as a user runs it: brc-readcount (C++ host over the C ABI) BAM -> text on /dev/null, one process,
    beside the reference binary on the same file."""
    from bam_readcount_b200 import build, synth_cb
    from oracle.oracle import REF_BIN, REF_SAMTOOLS, have_reference_binary
    if not have_reference_binary():
        return {"value": None, "error": "samtools of oracle/_ref missing: cannot write the sample BAM"}
    wd = tempfile.mkdtemp(prefix="brc_txt_")
    try:
        nblk = args.text_blocks
        info = synth_cb.write_sample_bam(spec, 0, 0, nblk, wd, REF_SAMTOOLS)
        n_bp = nblk * synth_cb.BLOCK_BP
        cli = build.CLI
        cmd = [cli, "-w", "0"] + CONFIGS[cfg_name]["argv"] + ["-f", info["fasta"], info["bam"], f"chr1:1-{n_bp}"]
        best, phases = None, None
        for _ in range(2):
            t0 = time.perf_counter()
            with open(os.devnull, "wb") as dn:
                pr = subprocess.run(cmd, stdout=dn, stderr=subprocess.PIPE, env=dict(os.environ, BRC_CLI_TIMING="1"))
            dt = time.perf_counter() - t0
            if pr.returncode != 0:
                return {"value": None, "error": f"brc-readcount exited {pr.returncode}"}
            if best is None or dt < best:
                best = dt
                phases = " | ".join(l.split("] ", 1)[1] for l in pr.stderr.decode("latin-1").splitlines() if l.startswith("[brc timing] ") and "window " not in l)
        ref_bp = min(n_bp, 100_000)
        s, dt = _run_procs([[REF_BIN, "-w", "0"] + CONFIGS[cfg_name]["argv"] + ["-f", info["fasta"], info["bam"], f"chr1:1-{ref_bp}"]])
        out = {"value": n_bp / best, "unit": UNIT, "wall_s": best, "sample_bp": n_bp, "bam_bytes": os.path.getsize(info["bam"]),
               "reference_one_process": s / dt, "host_phases": phases,
               "what": "brc-readcount BAM -> text to /dev/null, one process incl. start-up (CUDA context ~1 s); reference binary on the first "
               f"{ref_bp} bp of the same file"}
        try:
            out["compressed_span"] = e2e_compressed_span(cfg_name, spec, info, n_bp)
        except Exception as ex:
            out["compressed_span"] = {"value": None, "error": str(ex)[:200]}
        return out
    finally:
        shutil.rmtree(wd, ignore_errors=True)


def e2e_compressed_span(cfg_name, spec, info, n_bp):
    """SURVEY.md §8 f-2 end to end: the BAM's COMPRESSED BGZF blocks go to the GPU (brc_push_bam_span: inflate + framing + kernels
    on the device), the packed records come back.  H2D = compressed bytes."""
    import torch
    from bam_readcount_b200 import bamio
    from bam_readcount_b200.engine import Engine
    hdr, _ = None, None
    bai = bamio.BaiIndex(info["bam"] + ".bai")
    text = subprocess.check_output([os.path.join(ROOT, "oracle", "_ref", "samtools"), "view", "-H", info["bam"]], text=True)
    h = bamio.BamHeader(text, ["chr1"], [info["length"]])
    rg_lib = {rg: h.lib_of_rg(rg) for rg in h.rg_lb}
    flags = CONFIGS[cfg_name]["flags"]
    e = Engine(lib_names=h.lib_names, **flags)
    try:
        e.set_reference(0, "chr1", info["length"], spec.ref_host(0, 0, info["length"]), 0)
        win = 1_280_000
        spans = []
        for b in range(0, n_bp, win):
            sp = bamio.bam_span(info["bam"], bai, 0, max(b - 1, 0), min(b + win, n_bp), rg_lib)
            keep = torch.frombuffer(bytearray(sp["comp"]), dtype=torch.uint8).pin_memory()
            sp["comp"] = keep.numpy()
            spans.append((b, min(b + win, n_bp), sp, keep))
        times, h2d, d2h = [], 0, 0
        for it in range(3):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            hh = dd = 0
            for b, en, sp, _ in spans:
                e.reset()
                e.begin_region(0, b, en, False)
                e.push_bam_span(sp)
                e.end_region()
                e._check(e.lib.brc_compute(e.h))
                hh += len(sp["comp"])
                if it == 0:
                    dd += e.packed().nbytes()
            dt = time.perf_counter() - t0
            if it:
                times.append(dt)
            else:
                d2h = dd
            h2d = hh
        ms = 1000.0 * sum(times) / len(times)
        return {"value": n_bp / (ms / 1000.0), "unit": UNIT, "ms": ms, "h2d_bytes": h2d, "d2h_bytes": d2h, "windows": len(spans),
                "what": "compressed BGZF spans (pinned) -> brc_push_bam_span -> brc_compute; packed records back in host memory"}
    finally:
        e.close()


def run_deep(args):
    """C5: panel sites sharded over the ranks, `sites_per_window` sites per launch, reads generated in HBM."""
    import torch
    import torch.distributed as dist
    from bam_readcount_b200 import stream as st
    from bam_readcount_b200 import synth_cb
    from bam_readcount_b200.engine import CRegion, Engine

    cfg = CONFIGS["c5"]
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    spec = make_spec("c5", args)
    n_sites, per = args.c5_sites, args.c5_sites_per_window
    shards = st.plan_shards_weighted([1.0] * n_sites, world)
    s_lo, s_hi = shards[rank]
    wins = [(a, min(a + per, s_hi)) for a in range(s_lo, s_hi, per)]
    L = spec.deep_contig_len()
    flags = cfg["flags"]
    engs = [Engine(device=local, lib_names=LIBS, **flags) for _ in range(2)]
    dws = [synth_cb.DeviceWindow(spec, per * spec.depth, device) for _ in range(2)]
    # residency: the launches whose reads fit HBM next to the engines' buffers are generated once, before the timed region
    resident = {}
    if not args.no_resident:
        free_b, _ = torch.cuda.mem_get_info(device)
        budget = free_b - int(args.hbm_margin_gb * (1 << 30)) - 2 * per * spec.depth * 90     # the two engines' descriptor arrays
        for i, (a, b) in enumerate(wins):
            nr = (b - a) * spec.depth
            need = nr * synth_cb.DeviceWindow.bytes_per_read() + 4 * nr + (1 << 20)
            if budget < need:
                break
            dwr = synth_cb.DeviceWindow(spec, nr, device, scratch=dws[0].t["scratch"], with_region=True)
            dwr.fill(0, a, b, torch.cuda.current_stream().cuda_stream)
            resident[i] = dwr
            budget -= need
        torch.cuda.synchronize()
    streams = [torch.cuda.Stream(device=device) for _ in range(2)]
    done = [torch.cuda.Event() for _ in range(2)]
    ref_ascii = torch.empty(L + 64, dtype=torch.uint8, device=device)
    synth_cb.load().brc_synth_ref_device(C.byref(spec.c), 0, 0, L, ref_ascii.data_ptr(), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    for e in engs:
        e.set_reference_device(0, "chr1", L, 0, ref_ascii.data_ptr(), L, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()

    def regions_of(a, b):
        regs, slot = [], 0
        for k in range(a, b):
            p = spec.site_pos(k)
            i = k - a
            regs.append(CRegion(0, p, p + 1, 1, i * spec.depth, (i + 1) * spec.depth, slot, p - 1, 2))
            slot += 2
        return regs

    used = [False, False]

    def launch(i, a, b):
        h = i % 2
        if used[h]:
            done[h].synchronize()
        sp = streams[h].cuda_stream
        dw = resident.get(i)
        if dw is None:
            dw = dws[h]
            dw.fill(0, a, b, sp)
        engs[h].plan_device(regions_of(a, b), (b - a) * spec.depth, 65536)
        engs[h].run_device(dw.c_batch(), dw.t["region"].data_ptr(), sp)
        with torch.cuda.stream(streams[h]):
            done[h].record(streams[h])
        used[h] = True

    def one_pass():
        for i, (a, b) in enumerate(wins):
            launch(i, a, b)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        one_pass()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        one_pass()
    cur = torch.cuda.current_stream()
    for s in streams:
        cur.wait_stream(s)
    ev1.record()
    barrier()
    elapsed_ms = ev0.elapsed_time(ev1)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:
        last = [i % 2 for i in range(max(len(wins) - 2, 0), len(wins))]          # the handles of the last two launches, in order
        dump_outputs(args.dump_outputs, [(engs[h], streams[h]) for h in last])
    launches = len(wins) * args.steps * (3 + engs[0].launch_count())

    # stage times + parity of sampled sites (untimed)
    a, b = wins[0]
    used[0] = False
    launch(0, a, b)
    torch.cuda.synchronize()
    k0, k1 = engs[0].stage_ms(0), engs[0].stage_ms(1)
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    dws[0].fill(0, a, b, torch.cuda.current_stream().cuda_stream)
    g1.record()
    torch.cuda.synchronize()
    gen_ms = g0.elapsed_time(g1)
    res = engs[0].fetch_device_results(streams[0].cuda_stream)
    parity = {"checked": False}
    if not args.no_parity:
        from oracle.oracle import Oracle
        hb, _ = spec.window_host(0, a, min(a + args.c5_parity_sites, b))
        nchk = min(args.c5_parity_sites, b - a)
        ref = spec.ref_host(0, 0, L)
        o = Oracle(lib_names=LIBS, **flags)
        for i in range(nchk):
            p = spec.site_pos(a + i)
            o.region(hb, tid=0, beg=p, end=p + 1, contig="chr1", chrom_len=L, ref_seq=ref, ref_win_beg=0, site_list_mode=True,
                     read_lo=i * spec.depth, read_hi=(i + 1) * spec.depth)
        od = o.dump()
        ed = "".join(res.dump_range(hb, {0: (0, ref)}, i, spec.site_pos(a + i) - 1, spec.site_pos(a + i) + 1) for i in range(nchk))
        parity = {"checked": True, "identical": od == ed, "sites": nchk, "depth": spec.depth,
                  "what": "raw accumulator dump of the first sites of the rank's shard vs oracle/brc_oracle.c on the host-generated reads"}
    my_sites = s_hi - s_lo
    t = torch.tensor([elapsed_ms], device=device, dtype=torch.float64)
    u = torch.tensor([my_sites, launches, 1 if parity.get("identical", True) else 0], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        mn = u.clone()
        dist.all_reduce(mn, op=dist.ReduceOp.MIN)
        dist.all_reduce(u, op=dist.ReduceOp.SUM)
        par_all = bool(mn[2].item() >= 1)
    else:
        par_all = bool(parity.get("identical", True))
    if rank == 0:
        ms_per_step = float(t[0]) / args.steps
        tot_sites = float(u[0])
        events = tot_sites * spec.depth
        peak, peak_src = measured_peak_gbs()
        # algorithmic bytes (SURVEY.md §8d, C5): 245 B per read/event + outputs
        alg_win = (b - a) * spec.depth * 245
        line = {"metric": METRIC, "value": tot_sites / (ms_per_step / 1000.0), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32+f32 (f64 for one add)",
                "data": "synthetic",
                "config": {"workload": cfg["workload"], "flags": " ".join(cfg["argv"]), "sites": n_sites, "depth": spec.depth, "libraries": 8,
                           "sites_per_launch": per, "events_per_s": events / (ms_per_step / 1000.0), "shards": shards, "gen_ms_per_launch": gen_ms,
                           "inputs": f"{len(resident)} of rank 0's {len(wins)} launches resident in HBM before the timed region; the others are "
                                     "(re)generated in HBM by the counter-based generator inside it"},
                "roofline": {"bound": "hbm", "kernel": "deep_site_kernel + read_precompute_kernel, one launch of %d sites" % (b - a),
                             "achieved": alg_win / ((k0 + k1) / 1000.0) / 1e9, "peak": peak, "unit": "GB/s",
                             "frac": alg_win / ((k0 + k1) / 1000.0) / 1e9 / peak, "traffic": None, "peak_source": peak_src,
                             "algorithmic_bytes_per_launch": alg_win, "k0_ms": k0, "k1_ms": k1},
                "gpu_launches": int(u[1]), "parity": dict(parity, all_ranks_identical=par_all), "clocks": clocks}
        print(json.dumps(line))
    for e in engs:
        e.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c4", choices=sorted(CONFIGS))
    ap.add_argument("--contigs", type=int, default=0, help="c4: number of contigs (default 24)")
    ap.add_argument("--contig-blocks", type=int, default=0, help="contig length in 1280-bp generator blocks (default per config)")
    ap.add_argument("--e2e-windows", type=int, default=8, help="windows per rank in one e2e step (0 = skip e2e)")
    ap.add_argument("--e2e-handles", type=int, default=2, help="engine handles (host threads) the e2e caller keeps in flight")
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--parity-sites", type=int, default=20_000)
    ap.add_argument("--ref-sample", type=int, default=0, help="sites each reference process handles per step (0 = auto)")
    ap.add_argument("--text-blocks", type=int, default=8000, help="e2e_text sample size in 1280-bp blocks")
    ap.add_argument("--c5-sites", type=int, default=CONFIGS["c5"]["n_sites"])
    ap.add_argument("--c5-depth", type=int, default=CONFIGS["c5"]["depth"])
    ap.add_argument("--c5-sites-per-window", type=int, default=CONFIGS["c5"]["sites_per_window"])
    ap.add_argument("--c5-parity-sites", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e-text", action="store_true")
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--sec-msg-per-site", type=float, default=0.19, help="gather: pool records sent per site slot (fixed message size; C4 needs 0.152)")
    ap.add_argument("--reserve-ctas", type=int, default=0, help="N > 1: CTA slots pileup_kernel leaves free for the NCCL kernels of the gather")
    ap.add_argument("--no-resident", action="store_true", help="c4: regenerate every window inside the timed loop instead of keeping windows in HBM")
    ap.add_argument("--hbm-margin-gb", type=float, default=14.0, help="HBM left free when windows are kept resident")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of the results of the last step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        return reference_arm(args)
    if args.config == "c5":
        return run_deep(args)
    return run_wgs(args, args.config)


if __name__ == "__main__":
    sys.exit(main())
