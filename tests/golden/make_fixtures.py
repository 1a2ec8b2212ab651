#!/usr/bin/env python
"""Regenerates tests/golden/generated/* from the reference's own fixtures; the outputs are committed, so the tests need no
modkit checkout.   usage: make_fixtures.py <modkit v0.4.4 checkout>

hg002_updated.bam     = `modkit update-tags --mode ambiguous --no-implicit-probs` applied to
                        tests/resources/HG002_small.ch20._other.sorted.bam (tests/test_pileup.rs:161-175): Mm/Ml are
                        renamed MM/ML and the mode-less `C+m` header becomes `C+m?`; nothing else changes for pileup.
hg002_old_tags.bed    = the reference golden tests/resources/pileup-old-tags-regressiontest.methyl.bed
ecoli_reg.sorted.bam  = copy of the all-context, default-mode fixture (used with --force-allow-implicit vs the oracle)
"""
import os, shutil, sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(HERE)), "tools"))
import bamio  # noqa: E402

OUT = os.path.join(HERE, "generated")


def main():
    res = os.path.join(sys.argv[1], "tests", "resources", "")
    os.makedirs(OUT, exist_ok=True)
    b = bamio.Bam(res + "HG002_small.ch20._other.sorted.bam")

    def mm_fix(ty, payload):
        parts = []
        for p in payload[:-1].decode().split(";"):
            if not p:
                continue
            hd, _, rest = p.partition(",")
            if not hd.endswith("?") and not hd.endswith("."):
                hd += "?"
            parts.append(hd + (("," + rest) if rest else ""))
        return (b"MM", "Z", (";".join(parts) + ";").encode() + b"\x00")

    b.records = [bamio.replace_aux(r, {b"Mm": mm_fix, b"MM": mm_fix, b"Ml": lambda ty, p: (b"ML", ty, p)}) for r in b.records]
    b.write(os.path.join(OUT, "hg002_updated.bam"), level=9)
    shutil.copy(res + "pileup-old-tags-regressiontest.methyl.bed", os.path.join(OUT, "hg002_old_tags.bed"))
    shutil.copy(res + "ecoli_reg.sorted.bam", os.path.join(OUT, "ecoli_reg.sorted.bam"))
    shutil.copy(res + "ecoli_reg.sorted.bam.bai", os.path.join(OUT, "ecoli_reg.sorted.bam.bai"))
    for f in os.listdir(OUT):
        os.chmod(os.path.join(OUT, f), 0o644)


if __name__ == "__main__":
    main()
