"""`modkit pileup-hemi` without a GPU: the CPU restatement (tools/hemi_oracle.cpp) against the reference's two goldens
(tests/test_pileup_hemi.rs), its skip-set rule on a hand-made BAM, and the product CLI's argument errors, which are raised
before any device is opened."""
import os
import struct
import subprocess

import pytest

from conftest import GEN, ROOT

BAM = os.path.join(GEN, "duplex_hemi.bam")
REGION = "chr20:22,613,835-22,640,468"
CHR20_LEN = 64444167
WINDOW_START = 22600000
MODKIT = os.path.join(ROOT, "modkit_b200", "_build", "modkit")


@pytest.fixture(scope="session")
def hemi_oracle_exe():
    exe = os.path.join(ROOT, "tools", "_build", "hemi_oracle")
    srcs = [os.path.join(ROOT, "tools", "hemi_oracle.cpp")] + [os.path.join(ROOT, "oracle", f) for f in os.listdir(os.path.join(ROOT, "oracle")) if f.endswith(".hpp")]
    if not os.path.exists(exe) or any(os.path.getmtime(s) > os.path.getmtime(exe) for s in srcs):
        os.makedirs(os.path.dirname(exe), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-pthread", srcs[0], "-o", exe, "-lz"])
    return exe


@pytest.fixture(scope="session")
def chr20_fa(tmp_path_factory):
    """Full-length chr20 (the length in the BAM header): N outside the committed window, the window verbatim (soft-mask case
    kept), one sequence line, with its .fai."""
    window = open(os.path.join(GEN, "chr20_22600000_22660000.txt")).read().strip()
    fa = str(tmp_path_factory.mktemp("ref") / "chr20.fa")
    with open(fa, "w") as f:
        f.write(">chr20\n")
        f.write("N" * WINDOW_START)
        f.write(window)
        f.write("N" * (CHR20_LEN - WINDOW_START - len(window)))
        f.write("\n")
    with open(fa + ".fai", "w") as f:
        f.write("chr20\t%d\t7\t%d\t%d\n" % (CHR20_LEN, CHR20_LEN, CHR20_LEN + 1))
    return fa


def run_hemi_oracle(exe, args, bam, out):
    p = subprocess.run([exe] + list(args) + [bam, "-o", out], capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    return open(out).read()


GOLDEN_CASES = [
    (["--motif", "CG", "0", "--region", REGION, "--no-filtering", "--mixed-delim"], "duplex_hemi_nofilt.bed"),   # test_pileup_hemi_hm
    (["--cpg", "--region", REGION, "--mixed-delim"], "duplex_hemi.bed"),                                          # test_pileup_hemi_preset
]


@pytest.mark.parametrize("args,golden", GOLDEN_CASES, ids=["nofilt", "preset"])
def test_hemi_oracle_matches_reference_goldens(hemi_oracle_exe, chr20_fa, tmp_path, args, golden):
    got = run_hemi_oracle(hemi_oracle_exe, args + ["-r", chr20_fa], BAM, str(tmp_path / "o.bed"))
    assert got == open(os.path.join(GEN, golden)).read()


# ---- a hand-made BAM: one read without MM/ML spanning three intervals ------------------------------------------------------
SITES = [20, 60, 110, 150, 210, 250]          # CpG positions of the toy contig; no other C or G


def toy_contig():
    s = list(("ATTA" * 80)[:300])
    for p in SITES:
        s[p], s[p + 1] = "C", "G"
    return "".join(s)


def bam_record(name, pos, flag, cigar, seq, aux=b""):
    nt = {"=": 0, "A": 1, "C": 2, "G": 4, "T": 8, "N": 15}
    packed = bytearray((len(seq) + 1) // 2)
    for i, ch in enumerate(seq):
        packed[i // 2] |= nt[ch] << (4 if i % 2 == 0 else 0)
    ops = [(int(n), "MIDNSHP=X".index(o)) for n, o in cigar]
    nm = name.encode() + b"\0"
    core = struct.pack("<iiBBHHHiiii", 0, pos, len(nm), 60, 4680, len(ops), flag, len(seq), -1, -1, 0)
    return core + nm + b"".join(struct.pack("<I", n << 4 | o) for n, o in ops) + bytes(packed) + b"\xff" * len(seq) + aux


def mod_aux(mm, ml):
    return b"MMZ" + mm.encode() + b"\0" + b"MLBC" + struct.pack("<I", len(ml)) + bytes(ml)


def write_skip_case(tmp_path, with_diff=False):
    """(bam, fasta): read `good` carries C+m / G-m calls at every site; read `bare` has no MM/ML, starts at 10 and has a
    deletion over the first site, so its first column with a base in interval [0, 100) is 60. with_diff: read `diff` reads
    A,T over the site at 150 and carries A+a / T-a calls there (a pattern of primary base A: n_diff of the C rows)."""
    import bamio
    ref = toy_contig()
    fa = str(tmp_path / "toy.fa")
    open(fa, "w").write(">c1\n" + ref + "\n")
    open(fa + ".fai", "w").write("c1\t%d\t4\t%d\t%d\n" % (len(ref), len(ref), len(ref) + 1))
    n = len(SITES)
    good = bam_record("good", 0, 0, [(300, "M")], ref,
                      mod_aux("C+m?" + ",0" * n + ";G-m?" + ",0" * n + ";", [250, 10, 250, 10, 10, 250] + [250, 250, 10, 10, 250, 10]))
    bare = bam_record("bare", 10, 0, [(10, "M"), (1, "D"), (269, "M")], ref[10:20] + ref[21:290])
    out = bamio.Bam()
    out.header_text = b"@HD\tVN:1.6\tSO:coordinate\n@SQ\tSN:c1\tLN:300\n"
    out.refs = [("c1", 300)]
    out.records = [good, bare]
    if with_diff:
        seq = list(ref[140:160])
        seq[10], seq[11] = "A", "T"
        seq = "".join(seq)
        n_a, n_t = seq[:10].count("A"), seq[:11].count("T")
        out.records.append(bam_record("diff", 140, 0, [(20, "M")], seq, mod_aux("A+a?,%d;T-a?,%d;" % (n_a, n_t), [250, 250])))
    bam = str(tmp_path / ("diff.bam" if with_diff else "skip.bam"))
    out.write(bam)
    return bam, fa


SKIP_ARGS = ["--cpg", "--no-filtering", "-i", "100"]


def test_hemi_oracle_skip_set_one_nocall_per_interval(hemi_oracle_exe, tmp_path):
    bam, fa = write_skip_case(tmp_path)
    text = run_hemi_oracle(hemi_oracle_exe, SKIP_ARGS + ["-r", fa], bam, str(tmp_path / "o.bed"))
    rows = [line.split("\t") for line in text.splitlines()]
    assert sorted({int(r[1]) for r in rows}) == SITES
    nocall = {int(r[1]): int(r[17]) for r in rows}
    delete = {int(r[1]): int(r[14]) for r in rows}
    # intervals [0,100) [100,200) [200,300): one NoCall each, at the first column where `bare` has a base (20 is deleted)
    assert nocall == {20: 0, 60: 1, 110: 1, 150: 0, 210: 1, 250: 0}
    assert delete == {20: 1, 60: 0, 110: 0, 150: 0, 210: 0, 250: 0}
    # one (top, bottom) pattern per site from `good`: its two calls in order
    pats = {int(r[1]): r[3] for r in rows}
    assert pats == {20: "m,m,C", 60: "-,m,C", 110: "m,-,C", 150: "-,-,C", 210: "-,m,C", 250: "m,-,C"}


def test_hemi_oracle_n_diff(hemi_oracle_exe, tmp_path):
    bam, fa = write_skip_case(tmp_path, with_diff=True)
    text = run_hemi_oracle(hemi_oracle_exe, SKIP_ARGS + ["-r", fa], bam, str(tmp_path / "o.bed"))
    at = {r[3]: r for r in (line.split("\t") for line in text.splitlines()) if r[1] == "150"}
    assert set(at) == {"-,-,C", "a,a,A"}
    assert at["-,-,C"][16] == "1" and at["a,a,A"][16] == "1"       # n_diff: the other base's pattern calls


# ---- the product CLI: argument errors come before the device ---------------------------------------------------------
CLI_ERRORS = [
    (["-r", "ref.fa"], "either --cpg or a --motif must be provided for pileup-hemi"),
    (["-r", "ref.fa", "--motif", "CHG", "0"], "motif must be palindromic for pileup-hemi"),
    (["-r", "ref.fa", "--cpg", "--motif", "CG", "0"], "cannot be used with"),
    (["--cpg"], "--ref"),
    (["-r", "ref.fa", "--cpg", "--devices", "0,1"], "--devices"),
    (["-r", "ref.fa", "--cpg", "-f", "0.5"], "--sampling-frac 1.0"),
    (["-r", "ref.fa", "--cpg", "-f", "0.5", "--seed", "3"], "--seed"),
]


@pytest.mark.parametrize("args,message", CLI_ERRORS, ids=["no-motif", "not-palindromic", "cpg-and-motif", "no-ref", "devices", "frac", "seed"])
def test_hemi_cli_argument_errors(args, message):
    assert os.path.exists(MODKIT), "build() first"
    p = subprocess.run([MODKIT, "pileup-hemi"] + args + [BAM], capture_output=True, text=True)
    assert p.returncode == 2, p.stderr         # usage error: exit 2 (a device error would be exit 1)
    assert message in p.stderr
    assert "CUDA" not in p.stderr


# ---- the generator's --duplex option leaves every other output unchanged ------------------------------------------------
# sha256 of the inflated BAM stream written by the generator before --duplex existed (same arguments)
SYNTH_BASE = ["--contig", "c1:300000", "--contig", "c2:150000", "--coverage", "8", "--seed", "7", "--mean-len", "3000"]
SYNTH_BEFORE = [
    ([], "2ce53fef3a646547f378449c2b30ffe817a1714542c9dcf0272e99ed0eb6373f"),
    (["--mods", "hm", "--implicit", "--odd-records"], "8e861e91d6980a2216d67be65342bd468ef4864f7e71e2547630f5d1051985ae"),
    (["--mods", "hma", "--combined-hm", "--start-grid", "500"], "f1f9d4d188ad79db3eeb9f816bc15d897921644336a5fd6e86005f25d9c1546d"),
]


@pytest.mark.parametrize("extra,digest", SYNTH_BEFORE, ids=["m", "hm-implicit-odd", "hma-combined-grid"])
def test_synth_without_duplex_is_unchanged(synth_exe, tmp_path, extra, digest):
    import hashlib
    import bamio
    prefix = str(tmp_path / "g")
    subprocess.run([synth_exe, "--out", prefix] + SYNTH_BASE + extra, check=True, capture_output=True)
    assert hashlib.sha256(bamio.read_bgzf(prefix + ".bam")).hexdigest() == digest


def test_synth_duplex_lists(synth_exe, tmp_path):
    import bamio
    prefix = str(tmp_path / "d")
    subprocess.run([synth_exe, "--out", prefix, "--mods", "hm", "--duplex"] + SYNTH_BASE, check=True, capture_output=True)
    mm = [bamio.get_aux(r, b"MM") for r in bamio.Bam(prefix + ".bam").records[:50]]
    assert all(m.startswith(b"C+h?") and b";G-h?" in m and b";G-m?" in m for m in mm)
