#!/usr/bin/env python
"""`modkit pileup-hemi` measurement on one seeded --duplex contig (default 64.4 Mb at 40x, C+h/C+m and G-h/G-m lists):
    python tools/hemi_bench.py [--len 64444167] [--coverage 40] [--steps 10] [--dir /dev/shm/...] [--out result.json]
* the hemi pass (mkp_hemi_resident) on ONE resident chunk (the whole contig): CUDA-event ms per stage, averaged over --steps passes
  after 3 warm-up passes, and the library's launch count per pass;
* mkp_pileup_resident on the same chunk with the combine-strands bitmaps of CG (focus_pos = C, focus_neg = G), for comparison;
* the file -> bed wall time of `modkit pileup-hemi --cpg --no-filtering` (device ingest, output in the work directory);
* the CPU restatement (tools/_build/hemi_oracle, all host threads, same flags) on the first 8 Mb, as positions/s.
Prints one JSON object with the card name and its power limit. The genome is generated once into --dir."""
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        name, power = [x.strip() for x in out.splitlines()[0].split(",")]
        return name, power
    except Exception:
        return "unknown", "unknown"


def main():
    a = sys.argv[1:]
    length, cov, steps, work, out_json = 64444167, 40.0, 10, None, None
    i = 0
    while i < len(a):
        if a[i] == "--len": length = int(a[i + 1]); i += 2
        elif a[i] == "--coverage": cov = float(a[i + 1]); i += 2
        elif a[i] == "--steps": steps = int(a[i + 1]); i += 2
        elif a[i] == "--dir": work = a[i + 1]; i += 2
        elif a[i] == "--out": out_json = a[i + 1]; i += 2
        else: raise SystemExit("unknown argument " + a[i])
    work = work or "/dev/shm/mkb_hemi_%d_%g" % (length, cov)
    os.makedirs(work, exist_ok=True)
    prefix = os.path.join(work, "d")
    t = time.time()
    if not os.path.exists(prefix + ".bam.bai"):
        subprocess.run([os.path.join(ROOT, "tools", "_build", "synth_modbam"), "--out", prefix, "--contig", "syn1:%d" % length, "--coverage", str(cov),
                        "--mods", "hm", "--duplex", "--threads", str(min(96, os.cpu_count() or 8))], check=True, capture_output=True)
    gen_s = time.time() - t

    import numpy as np
    import modkit_b200
    ctx = modkit_b200.Context(0)
    bam = modkit_b200.Bam(prefix + ".bam", ctx=ctx)
    fpos, fneg = modkit_b200.motif_focus(prefix + ".fa", "syn1", 0, length, 100000, "CG:0", True)
    ctx.set_params(modkit_b200.make_params())            # --no-filtering: thresholds 0
    n_reads = bam.device_chunk(0, 0, length, focus=(fpos, fneg))
    starts = np.arange(0, length, 100000, dtype=np.uint32)     # (interval starts of the skip-set rule; -i 100000 without motif shifts)

    def passes(fn):
        for _ in range(3):
            fn()
        l0 = ctx.kernel_launches()
        acc = np.zeros(8)
        for _ in range(steps):
            st = fn()
            acc += np.array(list(st.kernel_ms))
        return acc / steps, (ctx.kernel_launches() - l0) / steps, st

    hemi_ms, hemi_launch, hst = passes(lambda: ctx.hemi_resident(1, starts))
    n_hemi_rows = int(hst.n_rows)
    pile_ms, pile_launch, pst = passes(lambda: ctx.pileup_resident())

    out_bed = os.path.join(work, "hemi.bed")
    exe = os.path.join(ROOT, "modkit_b200", "_build", "modkit")
    threads = str(min(64, os.cpu_count() or 8))
    t = time.time()
    subprocess.run([exe, "pileup-hemi", "--cpg", "--no-filtering", "-t", threads, "--quiet", "-r", prefix + ".fa", prefix + ".bam", "-o", out_bed], check=True)
    f2b_s = time.time() - t
    with open(out_bed, "rb") as f:
        f2b_rows = sum(1 for _ in f)

    oracle = os.path.join(ROOT, "tools", "_build", "hemi_oracle")
    win = min(8000000, length)
    t = time.time()
    subprocess.run([oracle, "--cpg", "--no-filtering", "-t", str(os.cpu_count() or 8), "--region", "syn1:0-%d" % win, "-r", prefix + ".fa", prefix + ".bam",
                    "-o", os.path.join(work, "oracle.bed")], check=True, capture_output=True)
    oracle_s = time.time() - t

    name, power = gpu_info()
    stage = lambda v, keys: {k: round(float(v[i]), 3) for i, k in keys}
    res = {
        "gpu": name, "power_limit": power, "contig_bp": length, "coverage": cov, "reads": int(n_reads), "generate_s": round(gen_s, 1),
        "hemi_pass_ms": stage(hemi_ms, [(0, "k_parse"), (1, "k_resolve"), (2, "column_rank"), (4, "k_hemi_pairs"), (5, "k_hemi_rows+scan"), (6, "host_sync"), (7, "total")]),
        "hemi_launches_per_pass": hemi_launch, "hemi_rows": n_hemi_rows, "hemi_columns": int(hst.n_hot),
        "pileup_pass_ms": stage(pile_ms, [(0, "k_parse"), (1, "k_resolve"), (2, "rank"), (4, "k_count_*"), (5, "k_rows"), (6, "host_sync"), (7, "total")]),
        "pileup_launches_per_pass": pile_launch, "pileup_rows": int(pst.n_rows),
        "file_to_bed_s": round(f2b_s, 3), "file_to_bed_rows": f2b_rows, "file_to_bed_positions_per_s": round(length / f2b_s),
        "oracle_window_bp": win, "oracle_s": round(oracle_s, 3), "oracle_positions_per_s": round(win / oracle_s), "oracle_threads": os.cpu_count(),
    }
    text = json.dumps(res)
    print(text)
    if out_json:
        with open(out_json, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
