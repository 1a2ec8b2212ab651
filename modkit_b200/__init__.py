"""modkit_b200 — B200-native `modkit pileup` hot path.

Python mirror of the host interface (ctypes over the in-tree C ABI, include/mkp.h + the mkh_* host API).
The reference seam is `process_region_batch` (src/pileup/mod.rs:684-716): reads of one genomic chunk go in,
`PileupFeatureCounts` rows come out. There is no CPU fallback: without the CUDA library or a GPU every entry
point raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("MODKIT_B200_LIB") or os.path.join(_HERE, "_build", "libmodkit_b200.so")   # env override: tuning variants only
_lib = None


class MkpError(RuntimeError):
    pass


class ReadHdr(C.Structure):
    _fields_ = [("ref_start", C.c_int32), ("l_seq", C.c_uint32), ("n_cigar", C.c_uint32), ("flags", C.c_uint32),
                ("off", C.c_uint64), ("len_ml", C.c_uint32), ("len_mm", C.c_uint32)]


class Params(C.Structure):
    _fields_ = [("default_threshold", C.c_float), ("base_threshold", C.c_float * 4), ("base_threshold_set", C.c_uint8 * 4),
                ("n_mod_thresholds", C.c_uint32), ("mod_code", C.c_uint32 * 16), ("mod_threshold", C.c_float * 16),
                ("numeric_mode", C.c_uint8), ("collapse_code", C.c_uint32), ("force_allow_implicit", C.c_uint8),
                ("edge_filter_on", C.c_uint8), ("edge_filter_inverted", C.c_uint8),
                ("edge_filter_start", C.c_uint32), ("edge_filter_end", C.c_uint32), ("max_depth", C.c_uint32)]


class Chunk(C.Structure):
    _fields_ = [("start", C.c_uint32), ("end", C.c_uint32), ("hdrs", C.POINTER(ReadHdr)), ("n_reads", C.c_uint32),
                ("heap", C.c_void_p), ("heap_bytes", C.c_uint64), ("focus_pos", C.c_void_p), ("focus_neg", C.c_void_p)]


class Stats(C.Structure):
    _fields_ = [("n_rows", C.c_uint64), ("n_hot", C.c_uint64), ("n_calls", C.c_uint64), ("n_reads_used", C.c_uint32),
                ("n_reads_skipped", C.c_uint32), ("n_states", C.c_uint32), ("device_error", C.c_uint32), ("kernel_ms", C.c_float * 8)]


ROW_DTYPE = np.dtype([("pos", "<u4"), ("code", "<u4"), ("strand", "u1"), ("primary_base", "u1"), ("reserved", "<u2"),
                      ("n_mod", "<u4"), ("n_canon", "<u4"), ("n_other", "<u4"), ("n_delete", "<u4"),
                      ("n_filtered", "<u4"), ("n_diff", "<u4"), ("n_nocall", "<u4")])
assert ROW_DTYPE.itemsize == 40

# mkp_hemi_row: one `modkit pileup-hemi` row; a half code is 0 for canonical ('-'), else a code point or 0x80000000|ChEBI
HEMI_ROW_DTYPE = np.dtype([("pos", "<u4"), ("primary_base", "u1"), ("reserved", "u1", (3,)), ("top_code", "<u4"), ("bottom_code", "<u4"),
                           ("count", "<u4"), ("n_canonical", "<u4"), ("n_other_pattern", "<u4"), ("n_delete", "<u4"),
                           ("n_fail", "<u4"), ("n_diff", "<u4"), ("n_nocall", "<u4")])
assert HEMI_ROW_DTYPE.itemsize == 44

MKP_SYMBOLS = ["mkp_create", "mkp_bind_host_thread", "mkp_destroy", "mkp_last_error", "mkp_set_params", "mkp_upload_chunk", "mkp_pileup_resident",
               "mkp_fetch_rows", "mkp_pileup_chunk", "mkp_sample_histogram", "mkp_sample_summary", "mkp_algorithmic_bytes", "mkp_kernel_launches",
               "mkp_device_memory", "mkp_bam_load", "mkp_bam_load_range", "mkp_bam_load_range_fd", "mkp_bam_records", "mkp_bam_chunk", "mkp_bam_tags", "mkp_bam_inflated", "mkp_fetch_chunk",
               "mkp_hemi_resident", "mkp_fetch_hemi_rows"]
MKH_SYMBOLS = ["mkh_pileup_main", "mkh_bam_open", "mkh_bam_close", "mkh_bam_n_refs", "mkh_bam_ref_name", "mkh_bam_ref_len",
               "mkh_bam_n_mapped", "mkh_bam_n_records", "mkh_pack_region", "mkh_packed_free", "mkh_packed_n_reads",
               "mkh_packed_hdrs", "mkh_packed_heap", "mkh_packed_heap_bytes", "mkh_packed_algorithmic_bytes", "mkh_format_rows",
               "mkh_motif_focus", "mkh_bam_open_device", "mkh_device_chunk", "mkh_bam_ingest_ms", "mkh_bam_total_records",
               "mkh_f32_display", "mkh_bam_partition_key", "mkh_bam_n_ranges", "mkh_pileup_main_sharded", "mkh_shard_plan",
               "mkh_bam_open_device_pieces", "mkh_bam_fetch", "mkh_summary_main", "mkh_sample_probs_main", "mkh_partition_key_of_cells", "mkh_bam_index_n_mapped", "mkh_pct2",
               "mkh_pileup_hemi_main"]

ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.POINTER(C.c_uint64), C.c_size_t, C.c_void_p)


def library_path():
    return _LIB_PATH


def load_library(build_if_missing=True):
    """dlopen the in-tree native library (building it with nvcc when absent). Never falls back to Python."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        if not build_if_missing:
            raise MkpError("native library missing: " + _LIB_PATH)
        from . import build as _build
        _build.build()
    lib = C.CDLL(_LIB_PATH)
    lib.mkp_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    lib.mkp_bind_host_thread.argtypes = [C.c_int]
    lib.mkp_destroy.argtypes = [C.c_void_p]
    lib.mkp_destroy.restype = None
    lib.mkp_last_error.argtypes = [C.c_void_p]
    lib.mkp_last_error.restype = C.c_char_p
    lib.mkp_set_params.argtypes = [C.c_void_p, C.POINTER(Params)]
    lib.mkp_upload_chunk.argtypes = [C.c_void_p, C.POINTER(Chunk)]
    lib.mkp_pileup_resident.argtypes = [C.c_void_p, C.POINTER(Stats)]
    lib.mkp_fetch_rows.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
    lib.mkp_pileup_chunk.argtypes = [C.c_void_p, C.POINTER(Chunk), C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.POINTER(Stats)]
    lib.mkp_sample_histogram.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_uint64)]
    lib.mkp_sample_summary.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.mkp_algorithmic_bytes.argtypes = [C.POINTER(Chunk), C.c_size_t]
    lib.mkp_algorithmic_bytes.restype = C.c_size_t
    lib.mkp_kernel_launches.argtypes = [C.c_void_p]
    lib.mkp_kernel_launches.restype = C.c_uint64
    lib.mkp_bam_load.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_uint64, C.c_void_p, C.c_size_t,
                                 C.POINTER(C.c_size_t), C.c_void_p]
    lib.mkp_bam_load_range.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t, C.c_uint64, C.c_uint64, C.c_void_p, C.c_size_t,
                                       C.POINTER(C.c_size_t), C.c_void_p]
    lib.mkp_device_memory.argtypes = [C.c_void_p, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    lib.mkh_pileup_main_sharded.argtypes = [C.c_int, C.POINTER(C.c_char_p), C.c_int, C.c_int, ALLREDUCE_FN, C.c_void_p, C.POINTER(C.c_double)]
    lib.mkh_shard_plan.argtypes = [C.c_char_p, C.c_uint32, C.c_int, C.c_void_p, C.c_void_p, C.c_uint64]
    lib.mkh_shard_plan.restype = C.c_int64
    lib.mkh_bam_open_device_pieces.argtypes = [C.c_char_p, C.c_void_p, C.c_void_p, C.c_uint32, C.POINTER(C.c_void_p)]
    lib.mkh_bam_fetch.argtypes = [C.c_char_p, C.c_uint32, C.c_int64, C.c_int64, C.c_void_p, C.c_uint64]
    lib.mkh_bam_fetch.restype = C.c_int64
    lib.mkp_bam_records.argtypes = [C.c_void_p, C.c_void_p]
    lib.mkp_bam_chunk.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p]
    lib.mkp_bam_tags.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_char_p, C.c_uint32, C.c_void_p]
    lib.mkp_bam_inflated.argtypes = [C.c_void_p, C.c_uint64, C.c_void_p, C.c_size_t]
    lib.mkp_fetch_chunk.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_uint32), C.c_void_p, C.POINTER(C.c_uint64)]
    lib.mkh_bam_open_device.argtypes = [C.c_char_p, C.c_void_p, C.POINTER(C.c_void_p)]
    lib.mkh_device_chunk.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
    lib.mkh_device_chunk.restype = C.c_int64
    lib.mkh_bam_ingest_ms.argtypes = [C.c_void_p, C.c_void_p]
    lib.mkh_bam_ingest_ms.restype = None
    lib.mkh_f32_display.argtypes = [C.c_float, C.c_char_p, C.c_int]
    lib.mkh_bam_partition_key.argtypes = [C.c_void_p, C.c_uint32, C.c_uint64, C.c_char_p, C.c_char_p, C.c_int]
    lib.mkh_pct2.argtypes = [C.c_float, C.c_char_p, C.c_int]
    lib.mkh_bam_index_n_mapped.argtypes = [C.c_char_p, C.c_uint32]
    lib.mkh_bam_index_n_mapped.restype = C.c_int64
    lib.mkh_partition_key_of_cells.argtypes = [C.c_void_p, C.c_uint32, C.c_char_p, C.c_int]
    lib.mkh_bam_n_ranges.argtypes = [C.c_void_p]
    lib.mkh_bam_n_ranges.restype = C.c_uint32
    lib.mkh_bam_total_records.argtypes = [C.c_void_p]
    lib.mkh_bam_total_records.restype = C.c_uint64
    lib.mkh_pileup_main.argtypes = [C.c_int, C.POINTER(C.c_char_p)]
    lib.mkh_summary_main.argtypes = [C.c_int, C.POINTER(C.c_char_p)]
    lib.mkh_pileup_hemi_main.argtypes = [C.c_int, C.POINTER(C.c_char_p)]
    lib.mkp_hemi_resident.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_uint32, C.POINTER(Stats)]
    lib.mkp_fetch_hemi_rows.argtypes = [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]
    lib.mkh_sample_probs_main.argtypes = [C.c_int, C.POINTER(C.c_char_p)]
    lib.mkh_bam_open.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_void_p)]
    lib.mkh_bam_close.argtypes = [C.c_void_p]
    lib.mkh_bam_close.restype = None
    lib.mkh_bam_n_refs.argtypes = [C.c_void_p]
    lib.mkh_bam_n_refs.restype = C.c_uint32
    lib.mkh_bam_ref_name.argtypes = [C.c_void_p, C.c_uint32]
    lib.mkh_bam_ref_name.restype = C.c_char_p
    lib.mkh_bam_ref_len.argtypes = [C.c_void_p, C.c_uint32]
    lib.mkh_bam_ref_len.restype = C.c_uint32
    lib.mkh_bam_n_mapped.argtypes = [C.c_void_p, C.c_uint32]
    lib.mkh_bam_n_mapped.restype = C.c_uint64
    lib.mkh_bam_n_records.argtypes = [C.c_void_p, C.c_uint32]
    lib.mkh_bam_n_records.restype = C.c_uint64
    lib.mkh_pack_region.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p)]
    lib.mkh_packed_free.argtypes = [C.c_void_p]
    lib.mkh_packed_free.restype = None
    lib.mkh_packed_n_reads.argtypes = [C.c_void_p]
    lib.mkh_packed_n_reads.restype = C.c_uint32
    lib.mkh_packed_hdrs.argtypes = [C.c_void_p]
    lib.mkh_packed_hdrs.restype = C.POINTER(ReadHdr)
    lib.mkh_packed_heap.argtypes = [C.c_void_p]
    lib.mkh_packed_heap.restype = C.c_void_p
    lib.mkh_packed_heap_bytes.argtypes = [C.c_void_p]
    lib.mkh_packed_heap_bytes.restype = C.c_uint64
    lib.mkh_packed_algorithmic_bytes.argtypes = [C.c_void_p]
    lib.mkh_packed_algorithmic_bytes.restype = C.c_uint64
    lib.mkh_format_rows.argtypes = [C.c_void_p, C.c_uint64, C.c_char_p, C.c_int, C.c_void_p, C.c_uint64]
    lib.mkh_format_rows.restype = C.c_uint64
    lib.mkh_motif_focus.argtypes = [C.c_char_p, C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_char_p, C.c_int, C.c_void_p, C.c_void_p]
    _lib = lib
    return lib


def pileup_main(args):
    """In-process `modkit pileup <args>`; returns the exit code (0 ok, 1 runtime error, 2 usage)."""
    lib = load_library()
    argv = (C.c_char_p * len(args))(*[str(a).encode() for a in args])
    return lib.mkh_pileup_main(len(args), argv)


def bind_host_thread(device):
    """Pin this thread (and threads started later) to the CPUs of the device's NUMA node. Returns 0 when bound."""
    return load_library().mkp_bind_host_thread(int(device))


def torch_allreduce(device=None):
    """Sum-all-reduce of a u64 vector over the default torch.distributed group (NCCL when `device` is a CUDA device,
    gloo on CPU): the transport of the two exchanges of an interval-sharded run."""
    import torch
    import torch.distributed as dist

    def fn(buf, n, _user):
        try:
            a = np.ctypeslib.as_array(buf, shape=(n,))
            t = torch.from_numpy(a.astype(np.int64))
            if device is not None:
                t = t.to(device)
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
            a[:] = t.cpu().numpy().astype(np.uint64)
            return 0
        except Exception as e:   # never let an exception cross the C boundary
            import sys
            print("allreduce failed: %r" % (e,), file=sys.stderr)
            return -1
    return fn


def pileup_main_sharded(args, rank, world, allreduce):
    """One rank of an interval-sharded `modkit pileup <args>` (every rank passes the same args plus its own --device).
    `allreduce(buf, n, user) -> 0` sums a u64 vector over the ranks in place (see torch_allreduce).
    Returns (exit code, stats dict)."""
    lib = load_library()
    argv = (C.c_char_p * len(args))(*[str(a).encode() for a in args])
    cb = ALLREDUCE_FN(allreduce) if allreduce is not None else C.cast(None, ALLREDUCE_FN)
    st = (C.c_double * 20)()
    rc = lib.mkh_pileup_main_sharded(len(args), argv, rank, world, cb, None, st)
    keys = ["total_s", "load_s", "thresholds_s", "gpu_s", "write_s", "rows_total", "positions_total", "rows_rank",
            "threshold_A", "threshold_C", "threshold_G", "threshold_T", "sampler_fetch_s", "intervals_s", "pack_s", "kernel_ms", "slice_s", "pass_s", "rowcopy_s"]
    return rc, dict(zip(keys, [float(x) for x in st]))


def bam_fetch(bam_path, tid, beg, end):
    """Offsets (inflated stream) of the records overlapping [beg,end) of tid, through the index (CPU only); tid None = the
    reads without coordinates."""
    lib = load_library()
    cap = 1 << 16
    while True:
        offs = np.zeros(cap, dtype=np.uint64)
        n = lib.mkh_bam_fetch(str(bam_path).encode(), 0xffffffff if tid is None else tid, beg, end, offs.ctypes.data, cap)
        if n < 0:
            raise MkpError("bam_fetch failed (%d)" % n)
        if n <= cap:
            return offs[:n].copy()
        cap = int(n)


def pct2(v):
    """The bedMethyl writer's two-decimal rendering of an f32 (== printf("%.2f")); CPU only."""
    buf = C.create_string_buffer(64)
    n = load_library().mkh_pct2(float(v), buf, 64)
    if n < 0:
        raise MkpError("pct2 failed")
    return buf.value.decode()


def bam_index_n_mapped(bam_path, tid):
    """Mapped reads of contig tid according to the index, as the device front end's index-only open reads it (CPU only)."""
    return int(load_library().mkh_bam_index_n_mapped(str(bam_path).encode(), tid))


def shard_plan(bam_path, interval_size, world):
    """[(rank, tid, start, end)] pieces of the interval-range shards the product uses for `world` ranks (CPU only)."""
    lib = load_library()
    cap = 4096
    while True:
        a = np.zeros(3 * cap, dtype=np.uint32)
        e = np.zeros(cap, dtype=np.uint32)
        n = lib.mkh_shard_plan(str(bam_path).encode(), interval_size, world, a.ctypes.data, e.ctypes.data, cap)
        if n < 0:
            raise MkpError("shard plan failed")
        if n <= cap:
            return [(int(a[3 * k]), int(a[3 * k + 1]), int(a[3 * k + 2]), int(e[k])) for k in range(n)]
        cap = int(n)


def summary_main(args):
    """In-process `modkit summary <args>` (pass --out FILE to get the report in a file); returns the exit code."""
    lib = load_library()
    argv = (C.c_char_p * len(args))(*[str(a).encode() for a in args])
    return lib.mkh_summary_main(len(args), argv)


def pileup_hemi_main(args):
    """In-process `modkit pileup-hemi <args>` (-o FILE, else stdout); returns the exit code (0 ok, 1 runtime error, 2 usage)."""
    lib = load_library()
    argv = (C.c_char_p * len(args))(*[str(a).encode() for a in args])
    return lib.mkh_pileup_hemi_main(len(args), argv)


def sample_probs_main(args):
    """In-process `modkit sample-probs <args>`; returns the exit code."""
    lib = load_library()
    argv = (C.c_char_p * len(args))(*[str(a).encode() for a in args])
    return lib.mkh_sample_probs_main(len(args), argv)


HDR_DTYPE = np.dtype([("ref_start", "<i4"), ("l_seq", "<u4"), ("n_cigar", "<u4"), ("flags", "<u4"), ("off", "<u8"), ("len_ml", "<u4"), ("len_mm", "<u4")])
MEMBER_DTYPE = np.dtype([("in_off", "<u8"), ("out_off", "<u8"), ("in_len", "<u4"), ("out_len", "<u4")])
REC_DTYPE = np.dtype([("off", "<u8"), ("size", "<u4"), ("tid", "<i4"), ("pos", "<i4"), ("end", "<i4"), ("flag", "<u4"), ("l_seq", "<u4")])
assert HDR_DTYPE.itemsize == 32 and MEMBER_DTYPE.itemsize == 24 and REC_DTYPE.itemsize == 32


class Bam:
    """A BAM file. With ctx=None the file is inflated and indexed on the host (zlib); with a Context the BGZF members are
    inflated, the record chain walked and the reads sliced on that GPU (mkp_bam_load / mkp_bam_chunk)."""

    def __init__(self, path, threads=4, ctx=None, pieces=None):
        self._lib = load_library()
        self._h = C.c_void_p()
        self._ctx = ctx
        if pieces is not None:
            # one rank of an interval-sharded run: only the byte ranges under the (tid, lo, hi) pieces go to the device
            a = np.ascontiguousarray(np.array(pieces, dtype=np.uint32).reshape(-1, 3))
            if self._lib.mkh_bam_open_device_pieces(str(path).encode(), ctx._h, a.ctypes.data, len(a), C.byref(self._h)):
                raise MkpError("cannot open BAM pieces on the device " + str(path))
        elif ctx is None:
            if self._lib.mkh_bam_open(str(path).encode(), threads, C.byref(self._h)):
                raise MkpError("cannot open BAM " + str(path))
        elif self._lib.mkh_bam_open_device(str(path).encode(), ctx._h, C.byref(self._h)):
            raise MkpError("cannot open BAM on the device " + str(path))

    def device_chunk(self, tid, start, end, focus=None):
        """Device ingest only: the reads overlapping [start,end) become the resident chunk of the context."""
        fp = fn = None
        if focus is not None:
            fp = np.ascontiguousarray(focus[0], dtype=np.uint32); fn = np.ascontiguousarray(focus[1], dtype=np.uint32)
        n = self._lib.mkh_device_chunk(self._h, tid, start, end, fp.ctypes.data if fp is not None else None, fn.ctypes.data if fn is not None else None)
        if n < 0:
            raise MkpError("device chunk failed")
        self._ctx._n_reads_hint = int(n)
        return int(n)

    @property
    def ingest_ms(self):
        ms = (C.c_float * 4)()
        self._lib.mkh_bam_ingest_ms(self._h, ms)
        return dict(zip(["h2d", "inflate", "walk", "total"], [float(x) for x in ms]))

    def partition_key(self, tid, i, tags):
        """--partition-tag key of the i-th record of contig tid (host-opened BAM): the key string, or None for NoKey."""
        buf = C.create_string_buffer(4096)
        rc = self._lib.mkh_bam_partition_key(self._h, tid, i, ":".join(tags).encode(), buf, 4096)
        if rc < 0:
            raise MkpError("partition key failed")
        return buf.value.decode() if rc == 1 else None

    @property
    def n_ranges(self):
        """Device ingest: 1 when the whole file is resident, else the number of byte ranges it is loaded in."""
        return int(self._lib.mkh_bam_n_ranges(self._h))

    @property
    def total_records(self):
        return int(self._lib.mkh_bam_total_records(self._h))

    def n_records(self, tid):
        return int(self._lib.mkh_bam_n_records(self._h, tid))

    def close(self):
        if self._h:
            self._lib.mkh_bam_close(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def refs(self):
        n = self._lib.mkh_bam_n_refs(self._h)
        return [(self._lib.mkh_bam_ref_name(self._h, i).decode(), self._lib.mkh_bam_ref_len(self._h, i)) for i in range(n)]

    def n_mapped(self, tid):
        return self._lib.mkh_bam_n_mapped(self._h, tid)

    def pack(self, tid, start, end):
        p = C.c_void_p()
        if self._lib.mkh_pack_region(self._h, tid, start, end, C.byref(p)):
            raise MkpError("pack_region failed")
        return Packed(self._lib, p, start, end)


class Packed:
    """Packed read blocks of one chunk (host memory owned by the native library)."""

    def __init__(self, lib, handle, start, end):
        self._lib, self._h, self.start, self.end = lib, handle, start, end
        self.n_reads = lib.mkh_packed_n_reads(handle)
        self.heap_bytes = lib.mkh_packed_heap_bytes(handle)
        self.algorithmic_bytes = lib.mkh_packed_algorithmic_bytes(handle)
        self._focus = None

    def set_focus(self, pos_bits, neg_bits):
        self._focus = (np.ascontiguousarray(pos_bits, dtype=np.uint32), np.ascontiguousarray(neg_bits, dtype=np.uint32))

    def chunk(self):
        ch = Chunk()
        ch.start, ch.end = self.start, self.end
        ch.hdrs = self._lib.mkh_packed_hdrs(self._h)
        ch.n_reads = self.n_reads
        ch.heap = self._lib.mkh_packed_heap(self._h)
        ch.heap_bytes = self.heap_bytes
        if self._focus is not None:
            ch.focus_pos = self._focus[0].ctypes.data
            ch.focus_neg = self._focus[1].ctypes.data
        return ch

    def headers(self):
        n = self.n_reads
        buf = C.cast(self._lib.mkh_packed_hdrs(self._h), C.POINTER(C.c_uint8 * (32 * n))).contents if n else b""
        return np.frombuffer(buf, dtype=HDR_DTYPE).copy() if n else np.zeros(0, dtype=HDR_DTYPE)

    def heap(self):
        n = self.heap_bytes
        if not n:
            return np.zeros(0, dtype=np.uint8)
        return np.frombuffer((C.c_uint8 * n).from_address(self._lib.mkh_packed_heap(self._h)), dtype=np.uint8).copy()

    def free(self):
        if self._h:
            self._lib.mkh_packed_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def f32_display(v):
    """Rust `{}` of an f32 as the host writes it (bedgraph fraction column, float aux values in partition keys)."""
    lib = load_library()
    buf = C.create_string_buffer(64)
    if lib.mkh_f32_display(float(np.float32(v)), buf, 64) < 0:
        raise MkpError("f32_display failed")
    return buf.value.decode()


def make_params(default_threshold=0.0, base_thresholds=None, mod_thresholds=None, numeric_mode=0, collapse_code=0,
                force_allow_implicit=False, edge_filter=None, edge_inverted=False):
    p = Params()
    p.default_threshold = default_threshold
    for b, v in (base_thresholds or {}).items():
        i = "ACGT".index(b)
        p.base_threshold[i] = v
        p.base_threshold_set[i] = 1
    for i, (code, v) in enumerate((mod_thresholds or {}).items()):
        p.mod_code[i] = ord(code) if isinstance(code, str) else (0x80000000 | int(code))
        p.mod_threshold[i] = v
        p.n_mod_thresholds = i + 1
    p.numeric_mode = numeric_mode
    p.collapse_code = ord(collapse_code) if isinstance(collapse_code, str) else collapse_code
    p.force_allow_implicit = 1 if force_allow_implicit else 0
    if edge_filter is not None:
        p.edge_filter_on = 1
        p.edge_filter_inverted = 1 if edge_inverted else 0
        p.edge_filter_start, p.edge_filter_end = edge_filter
    return p


class Context:
    """One GPU context (mkp_ctx). Raises when no CUDA device is usable: there is no CPU path."""

    def __init__(self, device=0):
        self._lib = load_library()
        self._h = C.c_void_p()
        rc = self._lib.mkp_create(device, C.byref(self._h))
        if rc:
            raise MkpError("mkp_create failed (%d): no usable CUDA device; this package has no CPU fallback" % rc)

    def _check(self, rc):
        if rc:
            raise MkpError(self._lib.mkp_last_error(self._h).decode())

    def set_params(self, params):
        self._check(self._lib.mkp_set_params(self._h, C.byref(params)))

    def upload(self, packed):
        ch = packed.chunk()
        self._check(self._lib.mkp_upload_chunk(self._h, C.byref(ch)))
        self._n_reads_hint = int(packed.n_reads)

    def pileup_resident(self):
        st = Stats()
        self._check(self._lib.mkp_pileup_resident(self._h, C.byref(st)))
        return st

    def fetch_rows(self):
        rows = C.c_void_p()
        n = C.c_size_t()
        self._check(self._lib.mkp_fetch_rows(self._h, C.byref(rows), C.byref(n)))
        if not n.value:
            return np.zeros(0, dtype=ROW_DTYPE)
        buf = (C.c_uint8 * (40 * n.value)).from_address(rows.value)
        return np.frombuffer(buf, dtype=ROW_DTYPE)   # view of ctx-owned pinned memory; copy() to keep

    def hemi_resident(self, offset, interval_starts):
        """The `pileup-hemi` pass on the resident chunk (uploaded with focus_pos = columns, focus_neg = partners)."""
        starts = np.ascontiguousarray(interval_starts, dtype=np.uint32)
        st = Stats()
        self._check(self._lib.mkp_hemi_resident(self._h, int(offset), starts.ctypes.data, len(starts), C.byref(st)))
        return st

    def fetch_hemi_rows(self):
        rows = C.c_void_p()
        n = C.c_size_t()
        self._check(self._lib.mkp_fetch_hemi_rows(self._h, C.byref(rows), C.byref(n)))
        if not n.value:
            return np.zeros(0, dtype=HEMI_ROW_DTYPE)
        buf = (C.c_uint8 * (HEMI_ROW_DTYPE.itemsize * n.value)).from_address(rows.value)
        return np.frombuffer(buf, dtype=HEMI_ROW_DTYPE)   # view of ctx-owned memory; copy() to keep

    def pileup_chunk(self, packed):
        ch = packed.chunk()
        rows = C.c_void_p()
        n = C.c_size_t()
        st = Stats()
        self._check(self._lib.mkp_pileup_chunk(self._h, C.byref(ch), C.byref(rows), C.byref(n), C.byref(st)))
        self._n_reads_hint = int(packed.n_reads)
        if not n.value:
            return np.zeros(0, dtype=ROW_DTYPE), st
        buf = (C.c_uint8 * (40 * n.value)).from_address(rows.value)
        return np.frombuffer(buf, dtype=ROW_DTYPE), st

    def sample_histogram(self, include_unaligned=False, take=None, want_contributes=False):
        hist = np.zeros((4, 1025), dtype=np.uint64)
        n = 0
        contrib = None
        inexact = C.c_uint64()
        take_p = None
        if take is not None:
            take = np.ascontiguousarray(take, dtype=np.uint8)
            take_p = take.ctypes.data
            n = len(take)
        if want_contributes:
            contrib = np.zeros(max(1, self._n_reads_hint), dtype=np.uint8)
        self._check(self._lib.mkp_sample_histogram(self._h, 1 if include_unaligned else 0, take_p, hist.ctypes.data,
                                                   contrib.ctypes.data if contrib is not None else None, C.byref(inexact)))
        return hist, contrib, inexact.value

    _n_reads_hint = 0

    @property
    def kernel_launches(self):
        return int(self._lib.mkp_kernel_launches(self._h))

    # ---- device ingest (mkp_bam_*) ----
    def bam_load(self, file_bytes, members, inflated_len, seeds):
        """file_bytes: the BGZF file (bytes / uint8 array); members: MEMBER_DTYPE array; seeds: sorted uint64 record starts."""
        fb = np.frombuffer(file_bytes, dtype=np.uint8) if not isinstance(file_bytes, np.ndarray) else file_bytes
        members = np.ascontiguousarray(members, dtype=MEMBER_DTYPE)
        seeds = np.ascontiguousarray(seeds, dtype=np.uint64)
        n = C.c_size_t()
        ms = (C.c_float * 4)()
        self._check(self._lib.mkp_bam_load(self._h, fb.ctypes.data, fb.size, members.ctypes.data, len(members), inflated_len,
                                           seeds.ctypes.data, len(seeds), C.byref(n), ms))
        self._n_records = n.value
        return n.value, [float(x) for x in ms]

    def bam_records(self):
        out = np.zeros(self._n_records, dtype=REC_DTYPE)
        if self._n_records:
            self._check(self._lib.mkp_bam_records(self._h, out.ctypes.data))
        return out

    def bam_inflated(self, off, length):
        out = np.zeros(length, dtype=np.uint8)
        self._check(self._lib.mkp_bam_inflated(self._h, off, out.ctypes.data, length))
        return out

    def bam_chunk(self, start, end, rec_ids, focus=None):
        ids = np.ascontiguousarray(rec_ids, dtype=np.uint32)
        fp = fn = None
        if focus is not None:
            fp = np.ascontiguousarray(focus[0], dtype=np.uint32); fn = np.ascontiguousarray(focus[1], dtype=np.uint32)
        self._check(self._lib.mkp_bam_chunk(self._h, start, end, ids.ctypes.data, len(ids), fp.ctypes.data if fp is not None else None,
                                            fn.ctypes.data if fn is not None else None))
        self._n_reads_hint = len(ids)

    TAG_CELL = 256      # MKP_TAG_CELL

    def bam_partition_keys(self, rec_ids, tags):
        """--partition-tag keys of device-resident records (mkp_bam_tags, four tags per call, + the host's key rule): list of str | None."""
        ids = np.ascontiguousarray(rec_ids, dtype=np.uint32)
        cells = np.zeros((len(ids), len(tags), self.TAG_CELL), dtype=np.uint8)
        for t0 in range(0, len(tags), 4):
            sub = tags[t0:t0 + 4]
            part = np.zeros((len(ids), len(sub), self.TAG_CELL), dtype=np.uint8)
            self._check(self._lib.mkp_bam_tags(self._h, ids.ctypes.data, len(ids), "".join(sub).encode(), len(sub), part.ctypes.data))
            cells[:, t0:t0 + len(sub), :] = part
        out, buf = [], C.create_string_buffer(8192)
        for i in range(len(ids)):
            row = np.ascontiguousarray(cells[i])
            rc = self._lib.mkh_partition_key_of_cells(row.ctypes.data, len(tags), buf, 8192)
            if rc < 0:
                raise RuntimeError("partition key too long")
            out.append(buf.value.decode() if rc == 1 else None)
        return out

    def fetch_chunk(self):
        """(headers, heap) of the resident chunk, copied back from the device (tests)."""
        n = C.c_uint32()
        hb = C.c_uint64(0)
        self._check(self._lib.mkp_fetch_chunk(self._h, None, C.byref(n), None, C.byref(hb)))
        hdrs = np.zeros(n.value, dtype=HDR_DTYPE)
        heap = np.zeros(hb.value, dtype=np.uint8)
        cap = C.c_uint64(hb.value)
        self._check(self._lib.mkp_fetch_chunk(self._h, hdrs.ctypes.data if n.value else None, C.byref(n), heap.ctypes.data if hb.value else None, C.byref(cap)))
        return hdrs, heap

    def close(self):
        if self._h:
            self._lib.mkp_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def format_rows(rows, chrom, mixed_delim=False):
    lib = load_library()
    rows = np.ascontiguousarray(rows)
    n = lib.mkh_format_rows(rows.ctypes.data, len(rows), chrom.encode(), 1 if mixed_delim else 0, None, 0)
    buf = C.create_string_buffer(n)
    lib.mkh_format_rows(rows.ctypes.data, len(rows), chrom.encode(), 1 if mixed_delim else 0, buf, n)
    return buf.raw[:n].decode()


def motif_focus(fasta, contig, start, end, interval_size=100000, motifs="CG:0", combine_strands=False):
    """Focus bitmaps (+ rule, - rule) over [start,end) on the reference's interval grid."""
    lib = load_library()
    nw = (end - start + 31) // 32
    pos = np.zeros(nw, dtype=np.uint32)
    neg = np.zeros(nw, dtype=np.uint32)
    if lib.mkh_motif_focus(str(fasta).encode(), contig.encode(), start, end, interval_size, motifs.encode(), 1 if combine_strands else 0,
                           pos.ctypes.data, neg.ctypes.data):
        raise MkpError("motif_focus failed")
    return pos, neg
