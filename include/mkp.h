/* mkp.h — C ABI of the B200-native `modkit pileup` hot path (device side).
 *
 * The reference (nanoporetech/modkit v0.4.4) has no FFI for this path; the seam this library
 * replaces is
 *     pub fn process_region_batch(&MultiChromCoordinates, bam_fp, &MultipleThresholdModCaller,
 *                                 &PileupNumericOptions, force_allow, combine_strands, max_depth,
 *                                 Option<&EdgeFilter>, Option<&Vec<SamTag>>)
 *         -> Vec<Result<ModBasePileup, String>>            (src/pileup/mod.rs:684-716)
 * called from src/pileup/subcommand.rs:739 and consumed by PileupWriter::write
 * (src/writers.rs:35-37, 159-183).  A Rust host binds these entry points with `extern "C"`
 * (see INTEGRATION.md); this repository's own host (C++/Python) uses the same entry points.
 *
 * Conventions: plain pointers and sizes only; no exceptions cross the boundary; every function
 * returns 0 on success and a negative code on failure (mkp_last_error gives the text); one
 * context per GPU / host thread; buffers are caller-owned unless stated.
 */
#ifndef MKP_H
#define MKP_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct mkp_ctx mkp_ctx;

/* ---- packed read blocks (what the host slices out of BAM records) -------------------------
 * One 32-byte header per read + one byte heap.  A read's heap block starts at `off`
 * (16-byte aligned) and holds, back to back:
 *     CIGAR   u32[n_cigar]          (BAM encoding: len<<4 | op, ops MIDNSHP=X)
 *     SEQ     u8[(l_seq+1)/2]       (BAM 4-bit encoding, "=ACMGRSVTWYHKDBN")
 *     ML      u8[len_ml]            (ML/Ml B:C array)
 *     MM      u8[len_mm]            (MM/Mm Z string without the NUL)
 * QNAME, QUAL and all other aux tags are not needed by the path and are not shipped.
 * Reads are in BAM (coordinate-sorted) order.
 */
typedef struct {
    int32_t  ref_start;   /* 0-based leftmost reference position (BAM pos)              */
    uint32_t l_seq;
    uint32_t n_cigar;
    uint32_t flags;       /* low 16 bits: BAM flag; high bits: MKP_RF_*                 */
    uint64_t off;         /* byte offset of the read's block in the heap                */
    uint32_t len_ml;
    uint32_t len_mm;
} mkp_read_hdr;

/* host-side tag lookup outcome (src/mod_bam.rs:1388-1470): MM/ML missing or of the wrong aux
 * type, or MN present and != l_seq  =>  the read yields no mod calls but still counts as a base */
#define MKP_RF_TAGS_INVALID (1u << 16)

/* ---- parameters: MultipleThresholdModCaller (src/threshold_mod_caller.rs:7-13) +
 *      PileupNumericOptions (src/pileup/mod.rs:667-671) + EdgeFilter (src/mod_bam.rs:1634-1639) */
#define MKP_MAX_MOD_THRESHOLDS 16
typedef struct {
    float    default_threshold;
    float    base_threshold[4];          /* A C G T */
    uint8_t  base_threshold_set[4];
    uint32_t n_mod_thresholds;
    uint32_t mod_code[MKP_MAX_MOD_THRESHOLDS];   /* char code point, or 0x80000000|ChEBI */
    float    mod_threshold[MKP_MAX_MOD_THRESHOLDS];
    uint8_t  numeric_mode;               /* 0 passthrough, 1 combine (--combine-mods), 2 collapse ReDistribute */
    uint32_t collapse_code;
    uint8_t  force_allow_implicit;
    uint8_t  edge_filter_on, edge_filter_inverted;
    uint32_t edge_filter_start, edge_filter_end;
    uint32_t max_depth;                  /* --max-depth (src/pileup/mod.rs:755-759 -> htslib bam_plp_set_maxcnt): a read that
                                            would make the column at its start position deeper than this is dropped from the
                                            pileup; 0 = no limit */
} mkp_params;

/* ---- one chunk of work: reads overlapping [start,end) of one contig -------------------------
 * focus_pos / focus_neg: optional bitmaps over [start,end) (bit i of word i/32 = position
 * start+i) holding the positions whose StrandRule admits the + / - tally
 * (FocusPositions::check_position, src/interval_chunks.rs:352-374).  NULL = AllPositions. */
typedef struct {
    uint32_t start, end;
    const mkp_read_hdr* hdrs;
    uint32_t n_reads;
    const uint8_t* heap;
    uint64_t heap_bytes;
    const uint32_t* focus_pos;
    const uint32_t* focus_neg;
} mkp_chunk;

/* ---- output row == PileupFeatureCounts (src/pileup/mod.rs:54-68), integers only ------------
 * valid_coverage = n_mod + n_canon + n_other; fraction_modified is formatted by the host. */
typedef struct {
    uint32_t pos;
    uint32_t code;        /* char code point, or 0x80000000|ChEBI                             */
    uint8_t  strand;      /* '+' or '-'                                                        */
    uint8_t  primary_base;/* 0..3 = A C G T                                                    */
    uint16_t reserved;
    uint32_t n_mod, n_canon, n_other, n_delete, n_filtered, n_diff, n_nocall;
} mkp_row;                /* 40 bytes */

typedef struct {          /* per-chunk counters, filled by mkp_pileup_* */
    uint64_t n_rows;
    uint64_t n_hot;           /* positions that received a counter slot            */
    uint64_t n_calls;         /* projected base-mod calls                           */
    uint32_t n_reads_used;    /* reads that produced mod calls (ReadCache "used")   */
    uint32_t n_reads_skipped; /* admitted reads without usable mod info (skip_set)  */
    uint32_t n_states;        /* distinct (primary base, mod code) pairs seen       */
    uint32_t device_error;    /* 0, or MKP_DERR_* bits (also turned into an error)  */
    float    kernel_ms[8];    /* CUDA-event ms: 0 parse 1 resolve 2 rank 3 (unused) 4 counters (k_count_bases, k_count_calls beside it) 5 rows 6 host sync/alloc 7 total
                                 (mkp_hemi_resident: 2 column rank, 4 k_hemi_pairs, 5 k_hemi_rows + scan) */
} mkp_stats;

#define MKP_DERR_TOO_MANY_STATES   1u   /* > 32 distinct (base,code) states                      */
#define MKP_DERR_TOO_MANY_LISTS    2u   /* > 16 MM lists in one read                             */
#define MKP_DERR_TOO_MANY_CODES    4u   /* > 4 codes at one read position                        */
#define MKP_DERR_IMPLICIT_MODE     8u   /* reserved (implicit '.'/default-mode fill is done on the device)      */
#define MKP_DERR_TOO_MANY_PATTERNS 16u  /* pileup-hemi: > 256 distinct (base, top, bottom) patterns in one chunk   */

/* ---- `modkit pileup-hemi` (src/pileup/duplex.rs, src/writers.rs:185-255) -------------------------------------------
 * One row per (position, primary base, pattern) == DuplexPatternCounts; valid coverage = count + n_other_pattern, the
 * percentage is formatted by the host. A half of the pattern is 0 for a canonical call ('-'), else a code point or
 * 0x80000000|ChEBI as in mkp_row. primary_base is the read base (0..3 = A C G T). */
typedef struct {
    uint32_t pos;
    uint8_t  primary_base;
    uint8_t  reserved[3];
    uint32_t top_code, bottom_code;
    uint32_t count, n_canonical, n_other_pattern, n_delete, n_fail, n_diff, n_nocall;
} mkp_hemi_row;           /* 44 bytes */

/* The hemi pass on the resident chunk. The chunk must carry two bitmaps: focus_pos = the hemi columns (the positive-strand
 * positions of the palindromic motif), focus_neg = their partner positions (column + offset); every partner must lie inside
 * [start, end) of the chunk. offset = MotifInfo::offset (reverse minus forward motif offset; may be negative).
 * interval_starts: the starts of the reference intervals the chunk covers, ascending (n_intervals >= 1, host memory): a read
 * without usable mod info adds one NoCall per interval, at its first column there. Rows stay on the device. */
int  mkp_hemi_resident(mkp_ctx* ctx, int32_t offset, const uint32_t* interval_starts, uint32_t n_intervals, mkp_stats* stats);
/* Rows of the last mkp_hemi_resident (host memory owned by ctx), sorted by position, primary base, top half, bottom half
 * (Canonical < code < ChEBI). */
int  mkp_fetch_hemi_rows(mkp_ctx* ctx, const mkp_hemi_row** rows, size_t* n_rows);

int  mkp_create(int device, mkp_ctx** out);
/* Pin the calling host thread (threads it creates later inherit the mask) to the CPUs of the NUMA node the device hangs off,
 * so that pinned staging buffers (first touch) and packer threads are local to the GPU's PCIe root. 0 = bound, 1 = no NUMA
 * information (nothing changed), <0 = error. */
int  mkp_bind_host_thread(int device);
void mkp_destroy(mkp_ctx* ctx);
const char* mkp_last_error(const mkp_ctx* ctx);   /* valid until the next call on ctx */
int  mkp_set_params(mkp_ctx* ctx, const mkp_params* params);

/* Copy a host chunk to the device (pinned or pageable host memory). The chunk stays resident
 * until the next mkp_upload_chunk / mkp_destroy. */
int  mkp_upload_chunk(mkp_ctx* ctx, const mkp_chunk* host_chunk);

/* Run the pileup kernels on the resident chunk. Rows stay on the device. */
int  mkp_pileup_resident(mkp_ctx* ctx, mkp_stats* stats);

/* Copy the rows of the last mkp_pileup_resident to host memory owned by ctx
 * (sorted by position, then strand '+' < '-', then code). */
int  mkp_fetch_rows(mkp_ctx* ctx, const mkp_row** rows, size_t* n_rows);

/* upload + pileup + fetch in one call: the drop-in for process_region_batch on host buffers. */
int  mkp_pileup_chunk(mkp_ctx* ctx, const mkp_chunk* host_chunk, const mkp_row** rows, size_t* n_rows,
                      mkp_stats* stats);

/* Threshold estimation support (src/thresholds.rs:118-156, src/mod_bam.rs:489-505): for the
 * resident chunk, histogram of the argmax probability of every call of the reads selected by
 * `take` (n_reads flags, host memory; NULL = all), per canonical base, bin = round(p*1024).
 * `contributes[i]` (optional, host memory, n_reads bytes) receives 1 when read i yielded >= 1
 * value.  hist is u64[4][1025]; `inexact` counts values that are not multiples of 1/1024. */
int  mkp_sample_histogram(mkp_ctx* ctx, int include_unaligned, const uint8_t* take,
                          uint64_t* hist, uint8_t* contributes, uint64_t* inexact);


/* `modkit summary` support (src/summarize.rs:117-252; SURVEY 8f-3): every base-modification call of the reads selected by `take`
 * (as in mkp_sample_histogram) is classed with the thresholds of mkp_set_params: a call that passes is counted under its
 * thresholded call, a call that fails under its arg-max call. Adds to table (u64[4][2][33]: canonical base A C G T, 0 pass / 1 fail,
 * 0 = canonical or 1 + state id) and reads_with (u64[4]: reads with calls on that base); obs (u32[4]) receives the state ids seen per
 * base (codes that were never the called state still get a row), states (u64[32]) the key of every state id of THIS call
 * (primary base << 32 | code; ~0 = unused) - state ids are only meaningful together with that array. */
int  mkp_sample_summary(mkp_ctx* ctx, int include_unaligned, const uint8_t* take, uint64_t* table, uint64_t* reads_with,
                        uint32_t* obs, uint64_t* states);

/* ---- BGZF / BAM ingest on the device (SURVEY §8f-1: the on-disk format step directly before the path) ----------
 * Replaces, for the records the path consumes, htslib's bgzf_read_block + inflate + bam_read1 behind
 * rust-htslib's bam::IndexedReader::{from_path, fetch} (src/pileup/mod.rs:732-743) and the tag lookup of
 * parse_raw_mod_tags (src/mod_bam.rs:1388-1470).  The host only walks the BGZF member headers (no inflate) and
 * turns BAI virtual offsets into seed offsets; inflate, record discovery and record slicing run on the GPU and the
 * packed chunk never exists in host memory.  CRC32 of the members is not verified. */
typedef struct {
    uint64_t in_off;      /* offset of the member's raw deflate payload in the file            */
    uint64_t out_off;     /* offset of its output in the inflated stream                        */
    uint32_t in_len;      /* payload bytes (BSIZE + 1 - 12 - XLEN - 8)                          */
    uint32_t out_len;     /* ISIZE                                                              */
} mkp_bgzf_member;

typedef struct {          /* one alignment record of the inflated stream                        */
    uint64_t off;         /* offset of its refID field                                          */
    uint32_t size;        /* block_size                                                         */
    int32_t  tid, pos;
    int32_t  end;         /* htslib bam_endpos: pos + reference length (1 without CIGAR)        */
    uint32_t flag;
    uint32_t l_seq;
} mkp_bam_rec;            /* 32 bytes */

/* Free / total bytes of the context's device (the ingest keeps the file and the inflated stream resident: callers
 * check that they fit and otherwise slice on the host and use mkp_upload_chunk). */
int  mkp_device_memory(mkp_ctx* ctx, size_t* free_bytes, size_t* total_bytes);

/* Copy the BGZF file to the device, inflate all members, walk the record chain.
 * seeds: sorted offsets (inflated stream) of known record starts, seeds[0] = first record; every segment between
 * two seeds is walked by its own thread, so more seeds = more parallelism (one seed is valid, only slow).
 * ms (optional, float[4]): copy stream busy, start -> last member inflated (the slabs of the file are copied while earlier
 * slabs are inflated), record walk, total. */
int  mkp_bam_load(mkp_ctx* ctx, const uint8_t* file, size_t file_len, const mkp_bgzf_member* members, size_t n_members,
                  uint64_t inflated_len, const uint64_t* seeds, size_t n_seeds, size_t* n_records, float* ms);
/* The same for a byte range of the file (one or several contigs of a coordinate-sorted BAM, so that files larger than the
 * device memory are processed range by range): `file` points at the first member of the range, member offsets and
 * seeds are relative to the range, and the record walk stops at walk_end (<= inflated_len: the offset of the first
 * record that belongs to the next range; the last members of a range may hold its first bytes). */
int  mkp_bam_load_range(mkp_ctx* ctx, const uint8_t* file, size_t file_len, const mkp_bgzf_member* members, size_t n_members,
                        uint64_t inflated_len, uint64_t walk_end, const uint64_t* seeds, size_t n_seeds, size_t* n_records, float* ms);
/* The same, with the file range [file_off, file_off + file_len) read from the descriptor fd (pread into pinned staging buffers: no
 * page of the file is mapped into the caller; member offsets are relative to file_off). */
int  mkp_bam_load_range_fd(mkp_ctx* ctx, int fd, uint64_t file_off, size_t file_len, const mkp_bgzf_member* members, size_t n_members,
                           uint64_t inflated_len, uint64_t walk_end, const uint64_t* seeds, size_t n_seeds, size_t* n_records, float* ms);
/* Record table in file order (n_records entries, host memory). */
int  mkp_bam_records(mkp_ctx* ctx, mkp_bam_rec* out);
/* Make the records rec_ids[0..n) (indices into the record table, file order) the resident chunk for [start,end):
 * the device-side equivalent of slicing them on the host + mkp_upload_chunk. */
int  mkp_bam_chunk(mkp_ctx* ctx, uint32_t start, uint32_t end, const uint32_t* rec_ids, uint32_t n,
                   const uint32_t* focus_pos, const uint32_t* focus_neg);
/* --partition-tag on the device front end (src/util.rs:670-688, src/pileup/mod.rs:629-646): the values of n_tags (<= 4 per call) two-letter
 * aux tags (`tags`: 2 * n_tags characters) of the records rec_ids[0..n). out: n * n_tags * MKP_TAG_CELL bytes, per (record, tag): [0] aux
 * type character (0 = absent or not a stringable type), [1] value length, [2..] the value (Z/H text, or the raw little-endian scalar).
 * A text longer than MKP_TAG_CELL - 3 bytes is an error. */
#define MKP_TAG_CELL 256
int  mkp_bam_tags(mkp_ctx* ctx, const uint32_t* rec_ids, uint32_t n, const char* tags, uint32_t n_tags, uint8_t* out);
/* Test / debug access: bytes of the inflated stream; headers and heap of the resident chunk
 * (hdrs: n_reads entries or NULL; heap: *heap_bytes capacity in, bytes out; or NULL to query sizes). */
int  mkp_bam_inflated(mkp_ctx* ctx, uint64_t off, uint8_t* dst, size_t len);
int  mkp_fetch_chunk(mkp_ctx* ctx, mkp_read_hdr* hdrs, uint32_t* n_reads, uint8_t* heap, uint64_t* heap_bytes);

/* SURVEY §8(d) algorithmic bytes of a chunk: sum over reads of 32 + 4 n_cigar + ceil(l_seq/2) + len_mm + len_ml,
 * plus 40 bytes per emitted row (roofline accounting only). */
size_t mkp_algorithmic_bytes(const mkp_chunk* chunk, size_t n_rows);
/* Number of kernels this context has launched since mkp_create (bench.py reports the difference over its timed region). */
uint64_t mkp_kernel_launches(const mkp_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* MKP_H */
