#!/usr/bin/env python
"""Regenerates the `modkit pileup-hemi` fixtures in tests/golden/generated/ from the reference's own test resources (the outputs
are committed, so the tests need no modkit checkout).   usage: make_hemi_fixtures.py <modkit v0.4.4 checkout>

duplex_hemi.bam(.bai)  = the records of tests/resources/duplex_modcalls_sort.bam that overlap the region of the hemi goldens
                         (chr20:22,613,835-22,640,468; 4 of its 53 reads), with QUAL blanked and every aux tag except MM/ML/MN
                         dropped (nothing else is read by the pileup), plus a BAI written here. The output of both golden runs
                         is unchanged: they take --region, and the threshold estimation of the preset run samples every read of
                         the region either way.
duplex_hemi.bed, duplex_hemi_nofilt.bed
                       = copies of the two goldens (tests/test_pileup_hemi.rs)
chr20_22600000_22660000.txt
                       = bases 22,600,000-22,660,000 of tests/resources/GRCh38_chr20.fa, soft-mask case kept, one line (the
                         65 MB FASTA is not committed; the tests rebuild a full-length chr20 around this window)
"""
import os
import shutil
import struct
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(HERE)), "tools"))
import bamio  # noqa: E402

OUT = os.path.join(HERE, "generated")
REGION = ("chr20", 22613835, 22640468)
WINDOW = (22600000, 22660000)
MEMBER = 0xff00             # bamio.Bam.write: raw bytes per BGZF member
KEEP_TAGS = (b"MM", b"ML", b"MN", b"Mm", b"Ml")


def ref_span(f):
    n = sum(c >> 4 for c in f["cigar"] if (c & 15) in (0, 2, 3, 7, 8))
    return f["pos"], f["pos"] + (n if n else 1)


def strip(r):
    f = bamio.rec_fields(r)
    o = f["aux_off"]
    keep = [r[s:e] for t, ty, s, e in bamio.iter_aux(r, o) if t in KEEP_TAGS]
    return r[:o - f["l_seq"]] + b"\xff" * f["l_seq"] + b"".join(keep)


def reg2bin(beg, end):
    end -= 1
    for shift, first in ((14, 4681), (17, 585), (20, 73), (23, 9), (26, 1)):
        if beg >> shift == end >> shift:
            return first + (beg >> shift)
    return 0


def write_bai(bam, path):
    """BAI (SAM spec 5.2) of a file written by bamio.Bam.write: member k holds raw bytes [k * MEMBER, (k + 1) * MEMBER)."""
    coff, data = [], open(path, "rb").read()
    o = 0
    while o < len(data):
        coff.append(o)
        o += struct.unpack_from("<H", data, o + 16)[0] + 1
    voff = lambda u: (coff[u // MEMBER] << 16) | (u % MEMBER) if u // MEMBER < len(coff) - 1 else coff[-1] << 16
    u = 4 + 4 + len(bam.header_text) + 4 + sum(8 + len(n.encode()) + 1 for n, _ in bam.refs)
    idx = [dict(bins={}, lin=[], beg=None, end=0, n_map=0, n_unmap=0) for _ in bam.refs]
    for r in bam.records:
        f = bamio.rec_fields(r)
        size = 4 + len(r)
        if f["tid"] >= 0:
            R = idx[f["tid"]]
            vb, ve = voff(u), voff(u + size)
            beg, end = ref_span(f)
            ch = R["bins"].setdefault(reg2bin(beg, end), [])
            if ch and ch[-1][1] >> 16 == vb >> 16:
                ch[-1][1] = ve
            else:
                ch.append([vb, ve])
            for w in range(beg >> 14, ((end - 1) >> 14) + 1):
                while len(R["lin"]) <= w:
                    R["lin"].append(0)
                if not R["lin"][w]:
                    R["lin"][w] = vb
            R["beg"] = vb if R["beg"] is None else min(R["beg"], vb)
            R["end"] = max(R["end"], ve)
            R["n_unmap" if f["flag"] & 4 else "n_map"] += 1
        u += size
    out = [b"BAI\x01", struct.pack("<I", len(bam.refs))]
    for R in idx:
        anyr = R["n_map"] + R["n_unmap"] > 0
        out.append(struct.pack("<I", len(R["bins"]) + (1 if anyr else 0)))
        for b in sorted(R["bins"]):
            out.append(struct.pack("<II", b, len(R["bins"][b])))
            out += [struct.pack("<QQ", *c) for c in R["bins"][b]]
        if anyr:
            out.append(struct.pack("<IIQQQQ", 37450, 2, R["beg"], R["end"], R["n_map"], R["n_unmap"]))
        lin = R["lin"]
        for w in range(1, len(lin)):
            if not lin[w]:
                lin[w] = lin[w - 1]
        out.append(struct.pack("<I", len(lin)))
        out += [struct.pack("<Q", v) for v in lin]
    out.append(struct.pack("<Q", 0))
    with open(path + ".bai", "wb") as fh:
        fh.write(b"".join(out))


def fasta_window(fa, contig, start, end):
    """bases [start, end) of one contig, through the .fai"""
    for line in open(fa + ".fai"):
        name, _, off, lb, lbytes = line.split("\t")[:5]
        if name != contig:
            continue
        off, lb, lbytes = int(off), int(lb), int(lbytes)
        out = []
        with open(fa, "rb") as f:
            pos = start
            while pos < end:
                row, col = divmod(pos, lb)
                n = min(lb - col, end - pos)
                f.seek(off + row * lbytes + col)
                out.append(f.read(n).decode())
                pos += n
        return "".join(out)
    raise KeyError(contig)


def main():
    res = os.path.join(sys.argv[1], "tests", "resources", "")
    os.makedirs(OUT, exist_ok=True)
    src = bamio.Bam(res + "duplex_modcalls_sort.bam")
    tid = [n for n, _ in src.refs].index(REGION[0])
    out = bamio.Bam()
    out.header_text, out.refs = src.header_text, src.refs
    for r in src.records:
        f = bamio.rec_fields(r)
        beg, end = ref_span(f)
        if f["tid"] == tid and beg < REGION[2] and end > REGION[1]:
            out.records.append(strip(r))
    path = os.path.join(OUT, "duplex_hemi.bam")
    out.write(path, level=9)
    write_bai(out, path)
    for f in ("duplex_hemi.bed", "duplex_hemi_nofilt.bed"):
        shutil.copy(res + f, os.path.join(OUT, f))
    with open(os.path.join(OUT, "chr20_%d_%d.txt" % WINDOW), "w") as f:
        f.write(fasta_window(res + "GRCh38_chr20.fa", REGION[0], WINDOW[0], WINDOW[1]) + "\n")
    for f in ("duplex_hemi.bam", "duplex_hemi.bam.bai", "duplex_hemi.bed", "duplex_hemi_nofilt.bed", "chr20_%d_%d.txt" % WINDOW):
        os.chmod(os.path.join(OUT, f), 0o644)


if __name__ == "__main__":
    main()
