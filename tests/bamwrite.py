"""TEST INFRASTRUCTURE — a BAM + BAI writer for ReadBatch fixtures (SAM spec §4.1 BGZF, §4.2 BAM, §5.2 BAI), so that the
tests build their coordinate-sorted input files without an external samtools.

Laid out the way htslib writes them: the header in BGZF blocks of its own, records packed into blocks of at most 0xff00
uncompressed bytes without crossing a block edge, integer tags in the smallest type that holds the value, chunks of consecutive
records per bin, the 16 kb linear index over mapped records, the pseudo-bin 37450 with the reference's offsets and counts.
"""
from __future__ import annotations

import dataclasses
import os
import struct
import zlib

import numpy as np

from bam_readcount_b200.batch import BAM_FUNMAP, TAG_ABSENT

BLOCK = 0xff00
EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")
META_BIN = 37450


def reg2bin(beg: int, end: int) -> int:
    end -= 1
    for shift, off in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return off + (beg >> shift)
    return 0


def _int_tag(tag: bytes, v: int) -> bytes:
    if v >= 0:
        for t, fmt, hi in ((b"C", "<B", 0xFF), (b"S", "<H", 0xFFFF)):
            if v <= hi:
                return tag + t + struct.pack(fmt, v)
        return tag + b"I" + struct.pack("<I", v)
    for t, fmt, lo in ((b"c", "<b", -0x80), (b"s", "<h", -0x8000)):
        if v >= lo:
            return tag + t + struct.pack(fmt, v)
    return tag + b"i" + struct.pack("<i", v)


class _Bgzf:
    def __init__(self, fh, level: int):
        self.fh, self.level, self.buf, self.coff = fh, level, bytearray(), 0

    def tell(self) -> int:
        return (self.coff << 16) | len(self.buf)

    def flush(self):
        if not self.buf:
            return
        co = zlib.compressobj(self.level, zlib.DEFLATED, -15)
        comp = co.compress(bytes(self.buf)) + co.flush()
        blk = (b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", len(comp) + 25) + comp +
               struct.pack("<II", zlib.crc32(self.buf) & 0xFFFFFFFF, len(self.buf)))
        self.fh.write(blk)
        self.coff += len(blk)
        self.buf = bytearray()

    def write_record(self, rec: bytes):
        if self.buf and len(self.buf) + len(rec) > BLOCK:
            self.flush()
        self.buf += rec

    def close(self):
        self.flush()
        self.fh.write(EOF)


def header_text(contigs, n_libs: int = 8, read_group: bool = True) -> str:
    """The header synth.write_sam writes."""
    t = "@HD\tVN:1.6\tSO:coordinate\n" + "".join(f"@SQ\tSN:{n}\tLN:{ln}\n" for n, ln in contigs)
    if read_group:
        t += "".join(f"@RG\tID:rg{i}\tSM:s\tLB:lib{i}\n" for i in range(n_libs))
    return t


def write_bam(path: str, batch, contigs, n_libs: int = 8, read_group: bool = True, level: int = 6, index: bool = True) -> str:
    """``batch`` (coordinate-sorted, every read placed) as a BAM with the records synth.write_sam would write, and its .bai."""
    n = batch.n_reads
    tid, pos, flag = batch.tid.tolist(), batch.pos.tolist(), batch.flag.tolist()
    mapq, lq, nm, sm, lib = batch.mapq.tolist(), batch.l_qseq.tolist(), batch.nm.tolist(), batch.sm.tolist(), batch.lib.tolist()
    co, so, qo = (x.astype(np.int64).tolist() for x in (batch.cigar_off, batch.seq_off, batch.qual_off))
    cig, seq, qual = batch.cigar.astype("<u4").tobytes(), batch.seq.tobytes(), batch.qual.tobytes()
    end = batch.ref_end().tolist()
    # the record's bin field spans the CIGAR's reference length (sam_parse1); the index uses bam_endpos (pos + 1 if unmapped)
    ops = batch.cigar & 0xF
    span = np.concatenate([[0], np.cumsum(np.where(np.isin(ops, (0, 2, 3, 7, 8)), batch.cigar >> 4, 0).astype(np.int64))])
    rlen = (span[batch.cigar_off[1:].astype(np.int64)] - span[batch.cigar_off[:-1].astype(np.int64)]).tolist()
    absent = int(TAG_ABSENT)
    text = header_text(contigs, n_libs, read_group).encode()
    hdr = b"BAM\1" + struct.pack("<i", len(text)) + text + struct.pack("<i", len(contigs))
    for name, ln in contigs:
        hdr += struct.pack("<i", len(name) + 1) + name.encode() + b"\0" + struct.pack("<i", ln)
    voffs = np.zeros((n, 2), dtype=np.uint64)
    with open(path, "wb") as fh:
        bg = _Bgzf(fh, level)
        bg.buf += hdr
        bg.flush()
        for i in range(n):
            name = (batch.qname[i] if batch.qname is not None else f"r{i}").encode() + b"\0"
            nc = co[i + 1] - co[i]
            b = reg2bin(pos[i], pos[i] + (rlen[i] if nc else 1))
            body = (struct.pack("<iiBBHHHiiii", tid[i], pos[i], len(name), mapq[i], b, nc, flag[i], lq[i], -1, -1, 0) + name +
                    cig[4 * co[i]:4 * co[i + 1]] + seq[so[i]:so[i + 1]] + qual[qo[i]:qo[i + 1]])
            if nm[i] != absent:
                body += _int_tag(b"NM", nm[i])
            if sm[i] != absent:
                body += _int_tag(b"SM", sm[i])
            if read_group and lib[i] != 0xFFFF:
                body += b"RGZrg%d\0" % lib[i]
            rec = struct.pack("<i", len(body)) + body
            bg.write_record(rec)
            voffs[i, 1] = bg.tell()
            voffs[i, 0] = voffs[i, 1] - len(rec)
        bg.close()
    if index:
        _write_bai(path + ".bai", len(contigs), tid, pos, end, flag, voffs)
    return path


def _write_bai(path, n_ref, tid, pos, end, flag, voffs):
    refs = [dict(bins={}, lin={}, first=None, last=0, mapped=0, unmapped=0) for _ in range(n_ref)]
    cur = None                                      # (ref, bin, chunk begin) of the open run of records
    for i in range(len(pos)):
        r = refs[tid[i]]
        beg_v, end_v = int(voffs[i, 0]), int(voffs[i, 1])
        b = reg2bin(pos[i], end[i])
        if cur is not None and cur[0] is r and cur[1] == b:
            cur[3] = end_v
        else:
            if cur is not None:
                cur[0]["bins"].setdefault(cur[1], []).append((cur[2], cur[3]))
            cur = [r, b, beg_v, end_v]
        if r["first"] is None:
            r["first"] = beg_v
        r["last"] = end_v
        if flag[i] & BAM_FUNMAP:
            r["unmapped"] += 1
        else:
            r["mapped"] += 1
            for w in range(pos[i] >> 14, ((end[i] - 1) >> 14) + 1):
                r["lin"].setdefault(w, beg_v)
    if cur is not None:
        cur[0]["bins"].setdefault(cur[1], []).append((cur[2], cur[3]))
    out = bytearray(b"BAI\1" + struct.pack("<i", n_ref))
    for r in refs:
        bins = {}
        for b, chunks in r["bins"].items():
            merged = []
            for c in sorted(chunks):
                if merged and c[0] >> 16 <= merged[-1][1] >> 16:          # same BGZF block: one chunk
                    merged[-1] = (merged[-1][0], max(merged[-1][1], c[1]))
                else:
                    merged.append(c)
            bins[b] = merged
        out += struct.pack("<i", len(bins) + (r["first"] is not None))
        for b in sorted(bins):
            out += struct.pack("<Ii", b, len(bins[b])) + b"".join(struct.pack("<QQ", *c) for c in bins[b])
        if r["first"] is not None:
            out += struct.pack("<IiQQQQ", META_BIN, 2, r["first"], r["last"], r["mapped"], r["unmapped"])
        n_intv = max(r["lin"]) + 1 if r["lin"] else 0
        lin, prev = [], r["first"] or 0
        for w in range(n_intv):                      # empty windows: the previous window's offset (hts_idx_finish)
            prev = r["lin"].get(w, prev)
            lin.append(prev)
        out += struct.pack("<i", n_intv) + struct.pack(f"<{n_intv}Q", *lin)
    out += struct.pack("<Q", 0)
    with open(path, "wb") as fh:
        fh.write(out)


def write_sample_bam(spec, contig: int, lo: int, hi: int, workdir: str, contig_name: str = "chr1", level: int = 6) -> dict:
    """ref.fa (+.fai) and s.bam (+.bai) of the generator's blocks / sites [lo, hi) — the files synth_cb.write_sample_bam
    makes — written here.  The FASTA covers the contig from 0 to the end of the window (+ 400 bp), the @SQ length."""
    from bam_readcount_b200 import synth, synth_cb
    end = (hi * synth_cb.BLOCK_BP if spec.mode == synth_cb.WGS else spec.site_pos(hi)) + 400
    if spec.mode == synth_cb.WGS:
        end = min(end, spec.contig_len)
    fa = os.path.join(workdir, "ref.fa")
    synth.write_fasta(fa, contig_name, np.frombuffer(spec.ref_host(contig, 0, end), dtype=np.uint8))
    batch, _ = spec.window_host(contig, lo, hi)
    batch = dataclasses.replace(batch, tid=np.zeros_like(batch.tid))
    bam = write_bam(os.path.join(workdir, "s.bam"), batch, [(contig_name, end)], n_libs=spec.n_libs, level=level)
    return dict(fasta=fa, bam=bam, length=end, contig=contig_name)
