#!/usr/bin/env python
"""bench.py — genomic positions/sec to bedMethyl for the `modkit pileup` hot path on B200 (strong scaling).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...      (N > 1, one rank per GPU)

Workload (config.workload): ONE fixed synthetic genome for every N (strong scaling) — 8 contigs, 515,553,336 bp in total
(8 x chr20; contig lengths in the proportions of hg38 chr1..chr8), 40x ONT-like reads with C+h?/C+m? MM/ML lists,
`modkit pileup --preset traditional --ref g.fa` (= --cpg --combine-strands --ignore h, BASELINE.json configs[3] scaled to what
one node generates in seconds), filter threshold estimated from sampled reads. The genome is cut into N contiguous
interval ranges of equal BAM weight (the product's own shard plan: BAI-weighted cuts on the reference-interval grid); rank r
loads only the BGZF byte range under its intervals. No data-path collective; the exchanges are the start-up sum of the
sampled-probability histograms and the output slice sizes (NCCL all-reduce through torch.distributed).

A step = one pass of the hot path over the whole genome (all ranks together): decode MM/ML -> project through the CIGAR ->
threshold -> count -> rows. `value` = device-resident throughput; `e2e` = the same through mkp_upload_chunk + mkp_pileup_resident +
mkp_fetch_rows (== mkp_pileup_chunk) on pinned HOST buffers, copies inside the timed region; `file_to_bed` = the whole product
(`modkit pileup`, sharded over the N GPUs): BAM file in the page cache -> bedMethyl text in /dev/shm, compared byte for byte
with the CPU restatement's bedMethyl of a window (`parity_checked_rows`).
`--impl reference` times the CPU restatement of the reference (oracle/, the Rust crate cannot be built here) on a bounded
window of the same genome with every host core.
`--dump-outputs DIR` writes what the timed path computed in its last step (see output_arrays) as DIR/<name>.npy; the genome is
generated from a fixed seed, so two builds run with the same arguments can be compared output for output.
bench.py compiles nothing and writes nothing under the tree (which may be read-only): it uses what build() left there.
"""
import argparse
import ctypes
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = 64_444_167                      # chr20
HG38 = [248_956_422, 242_193_529, 198_295_559, 190_214_555, 181_538_259, 170_805_979, 159_345_973, 145_138_636]   # chr1..chr8
N_CONTIGS = 8
COVERAGE = 40
MODS = "hm"
SEED = 20260924
INTERVAL = 100_000
CPU_WINDOW = 48_000_000                # bounded CPU sample: first 48 Mb of contig 1 (480 intervals of 100 kb)
E2E_SUB_BP = 8_000_000                 # e2e: sub-chunks pipelined over two contexts
PRESET = ["--preset", "traditional"]
DUMP_ROWS = 500_000                    # --dump-outputs: sampled rows of the last step (13 float64 arrays: 52 MB)
ROW_FIELDS = ["pos", "code", "strand", "primary_base", "n_mod", "n_canon", "n_other", "n_delete", "n_filtered", "n_diff", "n_nocall"]


def genome(scale=1.0):
    total = int(UNIT * N_CONTIGS * scale)
    lens = [max(INTERVAL, int(total * x / sum(HG38))) for x in HG38]
    return [("syn%d" % (i + 1), n) for i, n in enumerate(lens)]


def sh(cmd, **kw):
    return subprocess.run(cmd, check=True, capture_output=True, text=True, **kw)


def ensure_tools():
    """The genome generator and the CPU oracle as build() left them."""
    tools = (os.path.join(ROOT, "tools", "_build", "synth_modbam"), os.path.join(ROOT, "oracle", "_build", "modkit_oracle"))
    missing = [p for p in tools if not os.access(p, os.X_OK)]
    if missing:
        raise SystemExit("bench.py: %s missing; build first (python __graft_entry__.py)" % ", ".join(missing))
    return tools


def shared_dir(tag):
    base = "/dev/shm" if os.path.isdir("/dev/shm") and shutil.disk_usage("/dev/shm").free > 96 << 30 else tempfile.gettempdir()
    d = os.path.join(base, "modkit_b200_bench_%s" % tag)
    os.makedirs(d, exist_ok=True)
    return d


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self._stop = index, [], threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no-samples"]}
        sm = sorted(float(r[0]) for r in self.rows)
        reasons = []
        for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]):
            if any(r[3 + i].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "power_w_max": max(float(r[2]) for r in self.rows),
                "samples": len(self.rows), "reasons": reasons}


def gen_genome(synth, d, contigs, coverage, window=None, threads=None):
    """The genome BAM (all contigs), or - window=(name, W) - only the reads overlapping [0, W) of the first contig: the generator
    draws reads per 256 kb start tile from independent streams, so the window file holds exactly the same reads."""
    prefix = os.path.join(d, "win" if window else "g")
    cmd = [synth, "--out", prefix, "--coverage", str(coverage), "--mods", MODS, "--seed", str(SEED), "--level", "1",
           "--threads", str(threads or min(96, os.cpu_count() or 8))]
    for name, n in (contigs[:1] if window else contigs):      # contig streams are seeded by their index: contig 1 alone is the same contig
        cmd += ["--contig", "%s:%d" % (name, n)]
    if window:
        cmd += ["--region-only", "0-%d" % window]
    info = json.loads(sh(cmd).stdout)
    return prefix, info


def cpu_reference_run(oracle, prefix, contig, window, threads, threshold=None, out_bed=None):
    """One timed run of the CPU restatement over [0, window) of the first contig (same flags as the GPU arm);
    returns the oracle's timing dict (positions, pileup_s = the per-interval hot loop, total_s = file -> bedMethyl)."""
    with tempfile.TemporaryDirectory() as td:
        tj = os.path.join(td, "t.json")
        bed = out_bed or os.path.join(td, "o.bed")
        cmd = [oracle, "pileup", "-t", str(threads)] + PRESET + ["--ref", prefix + ".fa", "--region", "%s:0-%d" % (contig, window), "--timing-json", tj]
        if threshold is not None:
            cmd += ["--filter-threshold", "C:%.9g" % threshold]
        subprocess.run(cmd + [prefix + ".bam", bed], check=True, capture_output=True)
        return json.load(open(tj))


def median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def output_arrays(pieces, rows, sample, seed):
    """--dump-outputs: rows[i] are the rows (modkit_b200.ROW_DTYPE) a caller of the timed path receives for pieces[i] = (tid, lo, hi).
    Returns float64 arrays (positions exceed float32's integers): a seeded sample of at most `sample` rows of the concatenated
    output - every field, the contig and the row's index - and, for the whole output, each piece's row count and the CRC32 of its
    rows' fields."""
    import zlib
    import numpy as np
    from numpy.lib import recfunctions

    counts = np.array([len(r) for r in rows], dtype=np.int64)
    ends = np.cumsum(counts)
    idx = np.sort(np.random.default_rng(seed).choice(int(ends[-1]), size=min(sample, int(ends[-1])), replace=False))
    which = np.searchsorted(ends, idx, side="right")
    local = idx - (ends - counts)[which]
    picked = np.concatenate([r[local[which == i]] for i, r in enumerate(rows)])
    out = {"rows_" + f: picked[f].astype(np.float64) for f in ROW_FIELDS}
    out["rows_contig"] = np.array([p[0] for p in pieces], dtype=np.float64)[which]
    out["rows_index"] = idx.astype(np.float64)
    out["pieces"] = np.array(pieces, dtype=np.float64).reshape(-1, 3)
    out["piece_rows"] = counts.astype(np.float64)
    out["piece_crc32"] = np.array([zlib.crc32(recfunctions.repack_fields(r[ROW_FIELDS]).view(np.uint8)) for r in rows], dtype=np.float64)
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scale", type=float, default=1.0, help="(development) genome size relative to 8 x chr20")
    ap.add_argument("--coverage", type=float, default=COVERAGE)
    ap.add_argument("--keep", action="store_true")
    ap.add_argument("--workdir", default=None, help="(development) reuse/keep the generated workload in this directory")
    ap.add_argument("--skip-cpu", action="store_true", help="(development, A/B runs) leave cpu_baseline and the parity check out")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the timed path computed in its last step as DIR/<name>.npy (float64, at most 64 MB)")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    a.warmup = max(a.warmup, 3) if a.impl == "b200" else a.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    contigs = genome(a.scale)
    total_bp = sum(n for _, n in contigs)
    cpu_window = min(CPU_WINDOW, (contigs[0][1] // INTERVAL) * INTERVAL)
    workload = {"workload": "BASELINE configs[3] scaled: one synthetic genome of %d contigs, %d bp (8 x chr20; hg38 chr1-8 proportions), %gx ONT-like reads, C+h?/C+m? MM/ML, modkit pileup --preset traditional (--cpg --combine-strands --ignore h), estimated threshold (-p 0.1); the same genome for every N" % (len(contigs), total_bp, a.coverage),
                "genome_bp": total_bp, "contigs": len(contigs), "coverage": a.coverage, "mods": MODS, "interval_size": INTERVAL,
                "sharding": "interval ranges of equal BAM weight (BAI), one range per GPU; rank loads only its BGZF byte range",
                "l2_policy": "inputs (1.8 GB packed reads per 64 Mb) exceed the 126 MB L2; no explicit flush"}
    nproc = os.cpu_count() or 1
    tag = os.environ.get("MASTER_PORT", str(os.getpid())) + "_" + os.environ.get("TORCHELASTIC_RUN_ID", "solo")

    if a.impl == "reference":
        if rank != 0:
            return 0
        synth, oracle = ensure_tools()
        d = a.workdir or shared_dir("ref_" + tag)
        os.makedirs(d, exist_ok=True)
        try:
            prefix, info = gen_genome(synth, d, contigs, a.coverage, window=cpu_window)
            vals, walls, last = [], [], None
            for i in range(a.warmup + a.steps):
                last = cpu_reference_run(oracle, prefix, contigs[0][0], cpu_window, nproc)      # estimates its own threshold, like the reference
                if i >= a.warmup:
                    vals.append(last["positions"] / last["pileup_s"])
                    walls.append(last["positions"] / last["total_s"])
            value = median(vals)
            line = {"impl": "reference", "metric": "genomic positions/sec to bedMethyl", "value": value, "unit": "positions/s", "n_gpus": a.gpus,
                    "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * cpu_window / value, "higher_is_better": True, "scaling": "strong",
                    "vs_baseline": None, "dtype": "u32 counts (f32 probabilities)", "data": "synthetic", "config": workload,
                    "cpu_baseline": {"value": value, "unit": "positions/s", "cores": nproc, "kind": "port",
                                     "sample": "first %d bp of contig 1 of the same genome (%d reads, %d intervals of 100 kb, dynamic scheduling over %d threads); median of %d runs of the per-interval pileup phase of the C++ restatement of modkit 0.4.4 (reference not buildable: no Rust toolchain)" % (cpu_window, info["reads"], cpu_window // INTERVAL, nproc, len(vals)),
                                     "load_s": last["load_s"], "pileup_s": last["pileup_s"], "spread": [min(vals), max(vals)]},
                    "file_to_bed": {"value": median(walls), "unit": "positions/s", "what": "process start -> bedMethyl file closed (BAM inflate + threshold estimation + pileup + write), window BAM in the page cache"},
                    "e2e": {"value": value, "unit": "positions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
            print(json.dumps(line))
        finally:
            if not (a.keep or a.workdir):
                shutil.rmtree(d, ignore_errors=True)
        return 0

    import numpy as np
    import torch
    import torch.distributed as dist
    import modkit_b200

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    synth, oracle = ensure_tools()
    lib = modkit_b200.load_library(build_if_missing=False)
    # host threads and (first-touch) pinned buffers on the NUMA node of this rank's GPU
    numa = modkit_b200.bind_host_thread(local_rank)
    threads = max(4, min(64, len(os.sched_getaffinity(0)) // max(1, min(world, 4))))
    dev = torch.device("cuda", local_rank)
    d = a.workdir or shared_dir(tag)
    os.makedirs(d, exist_ok=True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    try:
        # ---- the genome (rank 0 generates it; every rank reads its own byte range of the same file)
        t0 = time.time()
        info_path = os.path.join(d, "g.info.json")
        if rank == 0:
            if not (a.workdir and os.path.exists(info_path)):
                prefix, info = gen_genome(synth, d, contigs, a.coverage)
                json.dump(info, open(info_path, "w"))
        barrier()
        prefix, info = os.path.join(d, "g"), json.load(open(info_path))
        t_gen = time.time() - t0

        # ---- this rank's shard: the product's plan (BAI-weighted cuts on the interval grid)
        t0 = time.time()
        plan = modkit_b200.shard_plan(prefix + ".bam", INTERVAL, world)
        mine = [(tid, lo, hi) for r, tid, lo, hi in plan if r == rank]
        ctx0 = modkit_b200.Context(local_rank)
        dbam = modkit_b200.Bam(prefix + ".bam", ctx=ctx0, pieces=mine)
        t_load = time.time() - t0
        ingest_ms = dbam.ingest_ms

        # ---- start-up: threshold from sampled reads of this shard; the collective = histogram all-reduce (NCCL).
        # (bench shortcut for the -n 10042 schedule: the reads over the first 2 Mb of every piece; the exact schedule is what the
        #  file_to_bed arm below and the parity tests run)
        params0 = modkit_b200.make_params(numeric_mode=2, collapse_code="h")
        ctx0.set_params(params0)
        hist = np.zeros((4, 1025), dtype=np.uint64)
        for tid, lo, hi in mine:
            dbam.device_chunk(tid, lo, min(hi, lo + 2_000_000))
            h, _, inexact = ctx0.sample_histogram()
            assert inexact == 0
            hist += h
        from modkit_b200 import sharding
        hist = sharding.allreduce_histogram(hist, device=dev)
        thr = float(sharding.percentile_from_histogram(hist[1], 0.1))
        params = modkit_b200.make_params(base_thresholds={"C": thr}, numeric_mode=2, collapse_code="h")

        # ---- resident chunks (one context per piece) and pinned host sub-chunks (e2e)
        t0 = time.time()
        keep_alive = []

        def pinned_chunk(hdrs, heap, start, end, fpos, fneg):
            ph = torch.empty(max(32, hdrs.nbytes), dtype=torch.uint8, pin_memory=True)
            pp = torch.empty(max(16, heap.nbytes), dtype=torch.uint8, pin_memory=True)
            ph.numpy()[:hdrs.nbytes] = hdrs.view(np.uint8)
            pp.numpy()[:heap.nbytes] = heap
            fp_s, fn_s = torch.from_numpy(np.ascontiguousarray(fpos)).pin_memory(), torch.from_numpy(np.ascontiguousarray(fneg)).pin_memory()
            c = modkit_b200.Chunk()
            c.start, c.end, c.n_reads, c.heap_bytes = start, end, len(hdrs), heap.nbytes
            c.hdrs = ctypes.cast(ph.data_ptr(), ctypes.POINTER(modkit_b200.ReadHdr))
            c.heap = pp.data_ptr()
            c.focus_pos, c.focus_neg = fp_s.data_ptr(), fn_s.data_ptr()
            keep_alive.append((ph, pp, fp_s, fn_s))
            alg = int(32 * len(hdrs) + 4 * int(hdrs["n_cigar"].sum()) + int(((hdrs["l_seq"].astype(np.int64) + 1) // 2).sum()) + int(hdrs["len_mm"].sum()) + int(hdrs["len_ml"].sum()))
            return c, hdrs.nbytes + heap.nbytes + 8 * (len(hdrs) + 1) + 2 * fp_s.numel() * 4, alg

        resident, subs = [], []
        reads_rank = 0
        for tid, lo, hi in mine:
            name = contigs[tid][0]
            fpos, fneg = modkit_b200.motif_focus(prefix + ".fa", name, lo, hi, INTERVAL, "CG:0", True)
            n = dbam.device_chunk(tid, lo, hi, focus=(fpos, fneg))
            hdrs, heap = ctx0.fetch_chunk()
            reads_rank += n
            c, _, alg = pinned_chunk(hdrs, heap, lo, hi, fpos, fneg)
            cx = modkit_b200.Context(local_rank)
            cx.set_params(params)
            assert lib.mkp_upload_chunk(cx._h, ctypes.byref(c)) == 0, lib.mkp_last_error(cx._h)
            resident.append((cx, alg, hi - lo))
            keep_alive.pop()                 # the piece-sized pinned copy is only needed for this upload
            del hdrs, heap, c
            # e2e sub-chunks on the interval grid
            nsub = max(1, -(-(hi - lo) // E2E_SUB_BP))
            bounds = [lo + (((hi - lo) * i // nsub) // INTERVAL) * INTERVAL for i in range(nsub)] + [hi]
            for i in range(nsub):
                s0, s1 = bounds[i], bounds[i + 1]
                if s1 <= s0:
                    continue
                w0, w1 = (s0 - lo) // 32, (s1 - lo + 31) // 32
                assert (s0 - lo) % 32 == 0
                dbam.device_chunk(tid, s0, s1)
                sh_, sp_ = ctx0.fetch_chunk()
                subs.append(pinned_chunk(sh_, sp_, s0, s1, fpos[w0:w1], fneg[w0:w1]))
        dbam.close()
        ctx0.close()
        t_pack = time.time() - t0
        ctxs = [modkit_b200.Context(local_rank), modkit_b200.Context(local_rank)]
        for cx in ctxs:
            cx.set_params(params)
        all_ctx = [r[0] for r in resident] + ctxs

        def launches():
            return sum(cx.kernel_launches for cx in all_ctx)

        # ---- value: device-resident passes over every resident chunk of the rank
        def resident_pass(acc=None):
            rows = 0
            for cx, _, _ in resident:
                st = cx.pileup_resident()
                rows += int(st.n_rows)
                if acc is not None:
                    acc += np.array(list(st.kernel_ms))
            return rows

        for _ in range(a.warmup):
            n_rows = resident_pass()
        stage = np.zeros(8)
        barrier()
        l0 = launches()
        with ClockSampler(local_rank) as clocks:
            t0 = time.perf_counter()
            for _ in range(a.steps):
                n_rows = resident_pass(stage)
            barrier()
            t_res = time.perf_counter() - t0
        stage /= a.steps
        l_res = launches() - l0
        if a.dump_outputs:
            # what mkp_fetch_rows hands the caller after the last timed mkp_pileup_resident (fetched outside the timed region)
            arrays = output_arrays(mine, [cx.fetch_rows() for cx, _, _ in resident], DUMP_ROWS // world, SEED + rank)
            os.makedirs(a.dump_outputs, exist_ok=True)
            for name, arr in arrays.items():
                np.save(os.path.join(a.dump_outputs, ("rank%d_" % rank if world > 1 else "") + name + ".npy"), arr)

        # ---- e2e: pinned host buffers -> rows on the host, every step; two contexts (two streams, two host threads) take
        # the sub-chunks alternately so that the H2D copy of one overlaps the kernels of the other. Every sub-chunk goes through
        # mkp_upload_chunk + mkp_pileup_resident + mkp_fetch_rows: the three calls mkp_pileup_chunk is made of.
        e2e_rows = [0]
        upload_lock = threading.Lock()

        def e2e_pass():
            counts = [0, 0]

            def worker(t, cx):
                rp, npp, stt = ctypes.c_void_p(), ctypes.c_size_t(), modkit_b200.Stats()
                for k in range(t, len(subs), 2):
                    with upload_lock:        # one upload at a time (full PCIe bandwidth)
                        rc = lib.mkp_upload_chunk(cx._h, ctypes.byref(subs[k][0]))
                    assert rc == 0, lib.mkp_last_error(cx._h)
                    rc = lib.mkp_pileup_resident(cx._h, ctypes.byref(stt))
                    assert rc == 0, lib.mkp_last_error(cx._h)
                    rc = lib.mkp_fetch_rows(cx._h, ctypes.byref(rp), ctypes.byref(npp))
                    assert rc == 0, lib.mkp_last_error(cx._h)
                    counts[t] += npp.value
            ths = [threading.Thread(target=worker, args=(t, cx)) for t, cx in enumerate(ctxs)]
            for th in ths:
                th.start()
            for th in ths:
                th.join()
            e2e_rows[0] = sum(counts)

        for _ in range(2):
            e2e_pass()
        barrier()
        l0 = launches()
        t0 = time.perf_counter()
        for _ in range(a.steps):
            e2e_pass()
        barrier()
        t_e2e = time.perf_counter() - t0
        l_e2e = launches() - l0
        h2d_bytes = sum(x[1] for x in subs)
        d2h_bytes = 40 * e2e_rows[0] + 64 * len(subs)
        for cx in all_ctx:
            cx.close()

        # ---- file_to_bed: the product, sharded over the N GPUs: BGZF file (page cache) -> bedMethyl text in /dev/shm.
        # In-process (CUDA context already created), twice; the second run is reported.
        out_bed = os.path.join(d, "out.bed")
        args = PRESET + ["--ref", prefix + ".fa", "-t", "32", "--device", str(local_rank), "--quiet", prefix + ".bam", out_bed]
        f2b = None
        for _ in range(2):
            barrier()
            t0 = time.perf_counter()
            rc, st_run = modkit_b200.pileup_main_sharded(args, rank, world, modkit_b200.torch_allreduce(dev) if world > 1 else None)
            assert rc == 0
            barrier()
            f2b = time.perf_counter() - t0

        # max over ranks
        times = torch.tensor([t_res, t_e2e, stage[7] * 1e-3, f2b], dtype=torch.float64, device="cuda")
        sums = torch.tensor([float(l_res + l_e2e), float(h2d_bytes), float(d2h_bytes), float(n_rows), float(reads_rank),
                             float(sum(r[1] for r in resident))] + [float(x) for x in stage], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(times, op=dist.ReduceOp.MAX)
            dist.all_reduce(sums, op=dist.ReduceOp.SUM)
        t_res, t_e2e, t_kern, f2b = [float(x) for x in times.cpu()]
        sums = [float(x) for x in sums.cpu()]
        n_launch, h2d_all, d2h_all, rows_all, reads_all, alg_in = sums[:6]
        stage_sum = np.array(sums[6:])          # per-stage ms summed over ranks (kernel time spent, all GPUs)
        value = total_bp * a.steps / t_res
        e2e = total_bp * a.steps / t_e2e

        if rank == 0:
            peaks = {}
            try:
                peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
            except Exception:
                pass
            peak = float(peaks.get("hbm_gbs", 6650.0))
            alg = alg_in + 40 * rows_all
            names = ["parse", "resolve", "rank", "unused", "count_calls+count_bases", "rows", "host_sync_alloc"]     # rank / host_sync_alloc are 0 on the focus-rank pass
            dom = int(np.argmax(stage_sum[:6]))
            # per-GPU rate of the dominant kernel: the bytes all GPUs' launches of it processed / the time they spent in it
            ach = alg / (stage_sum[dom] * 1e-3) / 1e9
            whole = alg / (stage_sum[7] * 1e-3) / 1e9
            # DRAM traffic per step (all launches of the kernel over the genome): one ncu capture of this workload, committed under
            # profiles/ (tools/profile_r02.sh); null for any other workload
            traffic, traffic_src, traffic_whole = None, None, None
            try:
                tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic_full.json")))
                kname = {"parse": "k_parse", "resolve": "k_resolve<0, 1>", "count_calls+count_bases": "k_count_bases", "rows": "k_rows<1>"}.get(names[dom])
                if tj.get("genome_bp") == total_bp and tj.get("coverage") == a.coverage and kname in tj["kernels"]:
                    traffic = int(tj["kernels"][kname]["dram_bytes_read"] + tj["kernels"][kname]["dram_bytes_write"])
                    traffic_whole = int(tj["whole_pass"]["dram_bytes"])
                    traffic_src = "profiles/r02_traffic_full.json (ncu dram__bytes_read.sum + dram__bytes_write.sum, summed over the kernel's launches of one pass over the genome)"
            except Exception:
                pass
            # ---- CPU baseline + parity of the bench's own output: the oracle on the first CPU_WINDOW bp of contig 1, same flags,
            # the threshold the product estimated; its bedMethyl must equal the product's file byte for byte
            cpu, parity_rows = None, None
            if not a.skip_cpu:
                wprefix, winfo = gen_genome(synth, d, contigs, a.coverage, window=cpu_window)
                runs = []
                obed = os.path.join(d, "oracle.bed")
                thr_file = st_run["threshold_C"]          # what the product estimated with the exact -n 10042 schedule
                assert thr_file > 0
                for i in range(3):
                    runs.append(cpu_reference_run(oracle, wprefix, contigs[0][0], cpu_window, nproc, threshold=thr_file, out_bed=obed))
                cpu_v = median([r["positions"] / r["pileup_s"] for r in runs])
                cpu_wall = median([r["positions"] / r["total_s"] for r in runs])
                cpu = {"value": cpu_v, "unit": "positions/s", "cores": nproc, "kind": "port",
                       "sample": "first %d bp of contig 1 of the same genome (%d intervals, dynamic scheduling over %d threads), same flags and threshold as the GPU arm; median of 3 runs of the per-interval pileup phase of the C++ restatement of modkit 0.4.4 (oracle/); BAM inflate+parse excluded (%.2f s)" % (cpu_window, cpu_window // INTERVAL, nproc, runs[-1]["load_s"]),
                       "file_to_bed": cpu_wall, "spread": [min(r["positions"] / r["pileup_s"] for r in runs), max(r["positions"] / r["pileup_s"] for r in runs)]}
                # rows of intervals that end before the window's last (clipped) interval are identical in both runs
                limit = cpu_window - INTERVAL - 1000
                name = contigs[0][0].encode()

                def rows_below(path):
                    out = []
                    with open(path, "rb") as f:
                        for ln in f:
                            c0 = ln.split(b"\t", 2)
                            if c0[0] != name:
                                if out:
                                    break
                                continue
                            if int(c0[1]) >= limit:
                                break
                            out.append(ln)
                    return out
                got, exp = rows_below(out_bed), rows_below(obed)
                assert len(exp) > 1000 and got == exp, "bench output differs from the oracle: %d vs %d rows" % (len(got), len(exp))
                parity_rows = len(exp)
            line = {"metric": "genomic positions/sec to bedMethyl", "value": value, "unit": "positions/s", "n_gpus": world, "steps": a.steps,
                    "warmup": a.warmup, "ms_per_step": 1e3 * t_res / a.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                    "dtype": "u32 counts (f32 probabilities)", "data": "synthetic", "config": workload, "impl": "b200",
                    "e2e": {"value": e2e, "unit": "positions/s", "h2d_bytes_per_step": int(h2d_all), "d2h_bytes_per_step": int(d2h_all),
                            "ms_per_step": 1e3 * t_e2e / a.steps,
                            "how": "sub-chunks of <= %d bp on the interval grid, 2 contexts/streams per GPU (H2D of one overlaps kernels of the other), pinned host memory on the GPU's NUMA node" % E2E_SUB_BP},
                    "file_to_bed": {"value": total_bp / f2b, "unit": "positions/s", "wall_s": f2b,
                                    "what": "modkit pileup --preset traditional sharded over %d GPU(s), in-process (CUDA context warm): BGZF file in the page cache -> H2D -> GPU inflate + record walk + slicing -> threshold estimation (10042 sampled reads, histogram all-reduce) -> pileup kernels -> strand combining + bedMethyl text -> file in /dev/shm; second of two runs, max over ranks" % world,
                                    "rank0_stages_s": st_run},
                    "parity_checked_rows": parity_rows,
                    "gpu_launches": int(n_launch),
                    "roofline": {"bound": "hbm", "kernel": names[dom], "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                                 "peak_source": "MEASURED_PEAKS.json (measured)" if peaks else "fallback 6650 GB/s", "traffic": traffic, "traffic_source": traffic_src,
                                 "algorithmic_bytes_per_step": int(alg), "kernel_ms_all_gpus": float(stage_sum[dom]),
                                 "whole_path": {"achieved": whole, "frac": whole / peak, "ms_all_gpus": float(stage_sum[7]), "traffic": traffic_whole}},
                    "stage_ms": {n: float(stage_sum[i]) for i, n in enumerate(names)},
                    "cpu_baseline": cpu,
                    "clocks": clocks.summary(),
                    "rows_per_step": int(rows_all), "reads": int(reads_all), "threshold_C": thr, "numa_bound": numa == 0,
                    "setup_s": {"generate": t_gen, "bam_load": t_load, "pack": t_pack, "ingest_ms_rank0": ingest_ms}}
            print(json.dumps(line))
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
    finally:
        if world > 1 and dist.is_initialized():
            try:
                dist.barrier()
            except Exception:
                pass
        if rank == 0 and not (a.keep or a.workdir):
            shutil.rmtree(d, ignore_errors=True)
    return 0


if __name__ == "__main__":
    sys.dont_write_bytecode = True     # no __pycache__ under the tree
    sys.exit(main())
