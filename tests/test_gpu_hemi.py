"""`modkit pileup-hemi` on the GPU: the product (pileup_hemi_main -> mkp_hemi_resident) against the reference's goldens and,
byte for byte, against the CPU restatement (tools/hemi_oracle.cpp) with the flag sets of DuplexModBamPileup."""
import os

import pytest

from conftest import GEN
from test_hemi_cpu import BAM, GOLDEN_CASES, REGION, SKIP_ARGS, chr20_fa, hemi_oracle_exe, run_hemi_oracle, write_skip_case  # noqa: F401

pytestmark = pytest.mark.gpu


def run_product(args, bam, out):
    import modkit_b200
    rc = modkit_b200.pileup_hemi_main(list(args) + ["--quiet", bam, "-o", out])
    return rc, (open(out).read() if os.path.isfile(out) else "")


def oracle_args(args):
    """the arguments without the product's own options (front end, chunk size): the output must not depend on them"""
    out, skip = [], False
    for a in args:
        if skip:
            skip = False
        elif a == "--gpu-chunk-bp":
            skip = True
        elif a != "--host-ingest":
            out.append(a)
    return out


def same_as_oracle(oracle, args, bam, tmp_path, min_rows=1):
    exp = run_hemi_oracle(oracle, oracle_args(args), bam, str(tmp_path / "o.bed"))
    rc, got = run_product(args, bam, str(tmp_path / "g.bed"))
    assert rc == 0
    assert got == exp
    assert exp.count("\n") >= min_rows
    return got


@pytest.mark.parametrize("args,golden", GOLDEN_CASES, ids=["nofilt", "preset"])
def test_gpu_hemi_reference_goldens(native_lib, chr20_fa, tmp_path, args, golden):
    rc, got = run_product(args + ["-r", chr20_fa], BAM, str(tmp_path / "g.bed"))
    assert rc == 0
    assert got == open(os.path.join(GEN, golden)).read()


FLAG_SETS = {
    "default-threshold": ["--cpg"],
    "tabs": ["--cpg", "--no-filtering"],
    "thresholds": ["--cpg", "--filter-threshold", "C:0.8", "--mod-thresholds", "h:0.9"],
    "combine-mods": ["--cpg", "--combine-mods", "--no-filtering"],
    "ignore-h": ["--cpg", "--ignore", "h"],
    "edge-filter": ["--cpg", "--edge-filter", "50", "--no-filtering"],
    "edge-filter-inverted": ["--cpg", "--edge-filter", "20,50", "--invert-edge-filter", "--no-filtering"],
    "cgcg0": ["--motif", "CGCG", "0", "--no-filtering"],
    "cgcg2": ["--motif", "CGCG", "2", "--no-filtering"],
    "mask": ["--cpg", "-k", "--no-filtering"],
    "mixed": ["--cpg", "--mixed-delim", "--no-filtering"],
    "small-intervals": ["--cpg", "-i", "1000", "--no-filtering"],
    "max-depth": ["--cpg", "--max-depth", "1", "-i", "2000", "--no-filtering"],
    "host-ingest": ["--cpg", "--host-ingest"],
}


SPARSE = {"edge-filter-inverted", "cgcg0", "cgcg2"}      # a handful of rows in the test region


@pytest.mark.parametrize("name", sorted(FLAG_SETS))
def test_gpu_hemi_flags_match_oracle(native_lib, hemi_oracle_exe, chr20_fa, tmp_path, name):
    same_as_oracle(hemi_oracle_exe, FLAG_SETS[name] + ["-r", chr20_fa, "--region", REGION], BAM, tmp_path, min_rows=1 if name in SPARSE else 50)


def test_gpu_hemi_whole_contig_and_include_bed(native_lib, hemi_oracle_exe, chr20_fa, tmp_path):
    same_as_oracle(hemi_oracle_exe, ["--cpg", "-r", chr20_fa, "--region", "chr20"], BAM, tmp_path, min_rows=200)
    bed = str(tmp_path / "inc.bed")
    with open(bed, "w") as f:
        f.write("chr20\t22614000\t22620000\n")
        f.write("chr20\t22625000\t22630000\tx\t0\t+\n")
    same_as_oracle(hemi_oracle_exe, ["--cpg", "--no-filtering", "-r", chr20_fa, "--include-bed", bed], BAM, tmp_path, min_rows=20)


def test_gpu_hemi_chunk_size_invariance(native_lib, chr20_fa, tmp_path):
    base = ["--cpg", "--no-filtering", "-r", chr20_fa, "--region", REGION]
    rc, a = run_product(base, BAM, str(tmp_path / "a.bed"))
    assert rc == 0
    for extra in (["--gpu-chunk-bp", "9973"], ["--gpu-chunk-bp", "9973", "-i", "997"]):
        for motif in ([], ["--motif", "CGCG", "2"]):
            args = base + extra
            if motif:
                args = [x for x in args if x != "--cpg"] + motif
                rc, ref = run_product([x for x in base if x != "--cpg"] + motif, BAM, str(tmp_path / "r.bed"))
                assert rc == 0
            else:
                ref = a
            rc, b = run_product(args, BAM, str(tmp_path / "b.bed"))
            assert rc == 0 and b == ref


def test_gpu_hemi_chebi_code_order(native_lib, hemi_oracle_exe, chr20_fa, tmp_path):
    """h rewritten to ChEBI 76792: rows order Code < ChEbi inside a pattern."""
    import bamio
    src = bamio.Bam(BAM)
    out = bamio.Bam()
    out.header_text, out.refs = src.header_text, src.refs
    fix = lambda ty, p: (b"MM", "Z", p[:-1].replace(b"C+h", b"C+76792").replace(b"G-h", b"G-76792") + b"\x00")
    out.records = [bamio.replace_aux(r, {b"MM": fix}) for r in src.records]
    bam = str(tmp_path / "chebi.bam")
    out.write(bam)
    got = same_as_oracle(hemi_oracle_exe, ["--cpg", "--no-filtering", "-r", chr20_fa, "--region", "chr20"], bam, tmp_path, min_rows=100)
    assert "76792," in got and ",76792," in got


@pytest.mark.parametrize("with_diff", [False, True], ids=["skip-set", "n-diff"])
def test_gpu_hemi_hand_made(native_lib, hemi_oracle_exe, tmp_path, with_diff):
    bam, fa = write_skip_case(tmp_path, with_diff)
    got = same_as_oracle(hemi_oracle_exe, SKIP_ARGS + ["-r", fa], bam, tmp_path, min_rows=6)
    if with_diff:
        assert any(line.split("\t")[1] == "150" and line.split("\t")[16] != "0" for line in got.splitlines())


# ---- seeded --duplex genomes (tools/synth_modbam.cpp) ---------------------------------------------------------------------
GENOME = ["--contig", "c1:400000", "--contig", "c2:250000", "--coverage", "20", "--seed", "20261017", "--mean-len", "4000", "--mods", "hm", "--duplex"]
SYNTH_CASES = {
    "default": ([], ["--cpg"]),
    "thresholds": ([], ["--cpg", "--filter-threshold", "C:0.8", "--mod-thresholds", "h:0.9"]),
    "combine-mods": ([], ["--cpg", "--combine-mods"]),
    "ignore-h": ([], ["--cpg", "--ignore", "h"]),
    "edge": ([], ["--cpg", "--edge-filter", "50", "--no-filtering"]),
    "edge-inverted": ([], ["--cpg", "--edge-filter", "20,50", "--invert-edge-filter", "--no-filtering"]),
    "implicit-allowed": (["--implicit"], ["--cpg", "--force-allow-implicit", "--no-filtering"]),
    "implicit-small-intervals": (["--implicit"], ["--cpg", "--no-filtering", "-i", "7000"]),
    "odd-records": (["--odd-records"], ["--cpg", "-i", "20000"]),
    "max-depth": (["--start-grid", "2000"], ["--cpg", "--max-depth", "6", "-i", "5000", "--no-filtering"]),
    "cgcg0": ([], ["--motif", "CGCG", "0", "--no-filtering"]),
    "cgcg2": ([], ["--motif", "CGCG", "2", "--no-filtering"]),
    "implicit-cgcg2": (["--implicit"], ["--motif", "CGCG", "2", "--force-allow-implicit", "--no-filtering", "--gpu-chunk-bp", "9973"]),
    "region-mask-mixed": ([], ["--cpg", "--region", "c2:20000-180000", "-k", "--mixed-delim"]),
    "small-chunks": ([], ["--cpg", "--no-filtering", "--gpu-chunk-bp", "9973", "-i", "997"]),
}
_genomes = {}


def duplex_genome(synth_exe, tmp_path_factory, extra):
    key = tuple(extra)
    if key not in _genomes:
        import subprocess
        prefix = str(tmp_path_factory.mktemp("duplex") / "g")
        subprocess.run([synth_exe, "--out", prefix] + GENOME + list(extra), check=True, capture_output=True)
        _genomes[key] = prefix
    return _genomes[key]


@pytest.mark.parametrize("name", sorted(SYNTH_CASES))
def test_gpu_hemi_synthetic_duplex(native_lib, hemi_oracle_exe, synth_exe, tmp_path_factory, tmp_path, name):
    gen, args = SYNTH_CASES[name]
    prefix = duplex_genome(synth_exe, tmp_path_factory, gen)
    got = same_as_oracle(hemi_oracle_exe, args + ["-r", prefix + ".fa"], prefix + ".bam", tmp_path, min_rows=100)
    if name == "default":
        pats = {line.split("\t")[3] for line in got.splitlines()}
        assert {"m,-,C", "-,m,C", "m,m,C", "m,h,C", "h,m,C", "-,-,C"} <= pats


def test_gpu_hemi_synthetic_chunk_invariance(native_lib, synth_exe, tmp_path_factory, tmp_path):
    prefix = duplex_genome(synth_exe, tmp_path_factory, [])
    base = ["--motif", "CGCG", "2", "--no-filtering", "-r", prefix + ".fa"]
    rc, a = run_product(base, prefix + ".bam", str(tmp_path / "a.bed"))
    rc2, b = run_product(base + ["--gpu-chunk-bp", "9973", "-i", "997"], prefix + ".bam", str(tmp_path / "b.bed"))
    assert rc == 0 and rc2 == 0 and a == b and a.count("\n") > 100
