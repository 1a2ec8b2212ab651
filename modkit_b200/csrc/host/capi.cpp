// Host C API used by the Python mirror (modkit_b200/__init__.py), tests and bench.py.
#include "pileup_hemi.hpp"

using namespace mkh;

struct mkh_bam { BamReader reader; };
struct mkh_packed { PackedChunk pc; };

extern "C" {

// In-process `modkit pileup`: returns the process exit code the reference would (0 ok, 1 error -> "> Error! ...").
int mkh_pileup_main(int argc, const char* const* argv) {
    PileupOptions o;
    std::string err;
    if (!parse_pileup_args(argc, argv, &o, &err)) { fprintf(stderr, "error: %s\n", err.c_str()); return 2; }
    RunSummary s;
    if (run_pileup_devices(o, &s, &err)) { fprintf(stderr, "> Error! %s\n", err.c_str()); return 1; }
    return 0;
}

// In-process `modkit pileup-hemi` (src/pileup/subcommand.rs:825-1514): argument errors exit 2 before any device is opened.
int mkh_pileup_hemi_main(int argc, const char* const* argv) {
    HemiOptions o;
    std::string err;
    if (!parse_hemi_args(argc, argv, &o, &err)) { fprintf(stderr, "error: %s\n", err.c_str()); return 2; }
    RunSummary s;
    if (run_pileup_hemi(o, &s, &err)) { fprintf(stderr, "> Error! %s\n", err.c_str()); return 1; }
    return 0;
}

// In-process `modkit summary` / `modkit sample-probs` (SURVEY 8f-3): the report goes to stdout, or to --out FILE.
static int sample_main(int argc, const char* const* argv, bool summary) {
    SampleOptions o;
    std::string err, out_path, text;
    if (!parse_sample_args(argc, argv, summary, &o, &out_path, &err)) { fprintf(stderr, "error: %s\n", err.c_str()); return 2; }
    if ((summary ? run_summary(o, &text, &err) : run_sample_probs(o, &text, &err))) { fprintf(stderr, "> Error! %s\n", err.c_str()); return 1; }
    if (out_path.empty()) fwrite(text.data(), 1, text.size(), stdout);
    else { FILE* f = fopen(out_path.c_str(), "w"); if (!f) { fprintf(stderr, "> Error! failed to make output file\n"); return 1; } fwrite(text.data(), 1, text.size(), f); fclose(f); }
    return 0;
}
int mkh_summary_main(int argc, const char* const* argv) { return sample_main(argc, argv, true); }
int mkh_sample_probs_main(int argc, const char* const* argv) { return sample_main(argc, argv, false); }

// One rank of an interval-sharded `modkit pileup` (SURVEY 8e): every rank is called with the same arguments (plus its own
// --device); `allreduce` sums a u64 vector over the ranks in place and returns 0 (NCCL through torch.distributed in
// bench.py / modkit_b200.pileup_main_sharded; any other transport works). It is called exactly twice per run, in the same
// order on every rank: the sampled-probability histograms (u64[4*1025 + 2]; thresholds.rs:118-156) and the output slice
// sizes (u64[world + 2]); with --include-unmapped a third, one-word exchange precedes them.
// out_stats (optional, double[20]): total_s, load_s, thresholds_s, gpu_s, write_s, rows (all ranks), positions (all ranks), rows of this
// rank, base thresholds A C G T (-1 = none), sampler fetch_s, intervals_s, pack_s, kernel_ms, slice_s, pass_s, rowcopy_s.
int mkh_pileup_main_sharded(int argc, const char* const* argv, int rank, int world, int (*allreduce)(uint64_t*, size_t, void*), void* user, double* out_stats) {
    PileupOptions o;
    std::string err;
    if (!parse_pileup_args(argc, argv, &o, &err)) { fprintf(stderr, "error: %s\n", err.c_str()); return 2; }
    if (rank < 0 || world < 1 || rank >= world || (world > 1 && !allreduce)) { fprintf(stderr, "error: bad rank/world\n"); return 2; }
    Collective c;
    c.rank = rank; c.world = world; c.allreduce_sum = allreduce; c.user = user;
    RunSummary s;
    if (run_pileup(o, &s, &err, &c)) { fprintf(stderr, "> Error! %s\n", err.c_str()); return 1; }
    trace_clock().mark(rank, "run returned (device + host buffers released)");
    if (out_stats) { out_stats[0] = s.total_s; out_stats[1] = s.load_s; out_stats[2] = s.threshold_s; out_stats[3] = s.gpu_s; out_stats[4] = s.write_s;
                     out_stats[5] = (double)s.rows_total; out_stats[6] = (double)s.positions_total; out_stats[7] = (double)s.rows;
                     for (int b = 0; b < 4; b++) out_stats[8 + b] = s.threshold_set[b] ? (double)s.thresholds[b] : -1.0;
                     out_stats[12] = s.fetch_s; out_stats[13] = s.interval_s; out_stats[14] = s.pack_s; out_stats[15] = s.kernel_ms;
                     out_stats[16] = s.slice_s; out_stats[17] = s.pass_s; out_stats[18] = s.rowcopy_s; }
    return 0;
}

// Shard plan of a BAM for `world` ranks (the cuts run_pileup uses; CPU only: header + index, no device): fills
// out[3 * k .. 3 * k + 2] = (rank, tid, start), end[k] per piece; returns the number of pieces, or -1.
int64_t mkh_shard_plan(const char* bam_path, uint32_t interval_size, int world, uint32_t* out_rank_tid_start, uint32_t* out_end, uint64_t cap) {
    try {
        BamReader bam;
        bam.open_device_index(bam_path, nullptr);
        std::vector<RefTarget> targets;
        for (uint32_t t = 0; t < bam.ref_names.size(); t++) targets.push_back({t, 0, bam.ref_lens[t], bam.ref_names[t]});
        std::vector<RefInterval> ivs = interval_grid(targets, interval_size, false, nullptr, nullptr);
        const std::vector<size_t> cuts = shard_cuts(bam, ivs, world);
        uint64_t n = 0;
        for (int r = 0; r < world; r++) {
            uint32_t tid = 0, lo = 0, hi = 0; bool open = false;
            auto flush = [&]() { if (!open) return; if (n < cap) { out_rank_tid_start[3 * n] = (uint32_t)r; out_rank_tid_start[3 * n + 1] = tid; out_rank_tid_start[3 * n + 2] = lo; out_end[n] = hi; } n++; open = false; };
            for (size_t i = cuts[r]; i < cuts[r + 1]; i++) {
                if (open && tid == ivs[i].tid && hi == ivs[i].start) { hi = ivs[i].end; continue; }
                flush();
                tid = ivs[i].tid; lo = ivs[i].start; hi = ivs[i].end; open = true;
            }
            flush();
        }
        return (int64_t)n;
    } catch (const std::exception& e) { fprintf(stderr, "mkh_shard_plan: %s\n", e.what()); return -1; }
}

int mkh_bam_open(const char* path, int threads, mkh_bam** out) {
    try { mkh_bam* b = new mkh_bam(); b->reader.open(path, threads); *out = b; return 0; }
    catch (const std::exception& e) { fprintf(stderr, "mkh_bam_open: %s\n", e.what()); return -1; }
}
// device ingest: inflate + record discovery on the GPU of `ctx` (include/mkp.h, mkp_bam_load)
int mkh_bam_open_device(const char* path, mkp_ctx* ctx, mkh_bam** out) {
    try { mkh_bam* b = new mkh_bam(); b->reader.open_device(path, ctx); *out = b; return 0; }
    catch (const std::exception& e) { fprintf(stderr, "mkh_bam_open_device: %s\n", e.what()); return -1; }
}
// the same for one rank of an interval-sharded run: only the byte ranges under the pieces (tid, lo, hi)[n] are loaded
int mkh_bam_open_device_pieces(const char* path, mkp_ctx* ctx, const uint32_t* tid_lo_hi, uint32_t n, mkh_bam** out) {
    try {
        mkh_bam* b = new mkh_bam();
        b->reader.open_device_index(path, ctx);
        std::vector<BamReader::Piece> pieces;
        for (uint32_t i = 0; i < n; i++) pieces.push_back({tid_lo_hi[3 * i], tid_lo_hi[3 * i + 1], tid_lo_hi[3 * i + 2]});
        b->reader.load_pieces(pieces);
        *out = b;
        return 0;
    } catch (const std::exception& e) { fprintf(stderr, "mkh_bam_open_device_pieces: %s\n", e.what()); return -1; }
}
// Host-side region fetch through the index (CPU only; the sampler's candidate source): offsets (inflated stream) of the records
// overlapping [beg,end) of tid, in file order. Returns the count (offsets beyond cap are not stored), or -1.
int64_t mkh_bam_fetch(const char* path, uint32_t tid, int64_t beg, int64_t end, uint64_t* offs, uint64_t cap) {
    try {
        BamReader r;
        r.open_device_index(path, nullptr);
        if (!r.have_index()) return -2;
        BamReader::FetchCursor c = tid == 0xffffffffu ? r.fetch_unplaced_begin() : r.fetch_begin(tid, beg, end);
        std::vector<RecRef> recs;
        while (!c.done) r.fetch_more(c, 4096, [](const RecRef&) { return true; }, &recs);
        for (size_t i = 0; i < recs.size() && i < cap; i++) offs[i] = recs[i].off;
        return (int64_t)recs.size();
    } catch (const std::exception& e) { fprintf(stderr, "mkh_bam_fetch: %s\n", e.what()); return -1; }
}
// the reads overlapping [start,end) of tid become the resident chunk of the ingest context; returns the read count or -1
int64_t mkh_device_chunk(const mkh_bam* b, uint32_t tid, uint32_t start, uint32_t end, const uint32_t* focus_pos, const uint32_t* focus_neg) {
    try {
        std::vector<RecRef> recs;
        b->reader.ensure_tid(tid);
        b->reader.for_overlapping(tid, start, end, [&](const RecRef& r) { recs.push_back(r); });
        return (int64_t)device_chunk(b->reader, recs, start, end, focus_pos, focus_neg);
    } catch (const std::exception& e) { fprintf(stderr, "mkh_device_chunk: %s\n", e.what()); return -1; }
}
void mkh_bam_ingest_ms(const mkh_bam* b, float* ms) { for (int i = 0; i < 4; i++) ms[i] = b->reader.ingest_ms[i]; }
uint32_t mkh_bam_n_ranges(const mkh_bam* b) { return (uint32_t)b->reader.n_ranges(); }
uint64_t mkh_bam_total_records(const mkh_bam* b) { uint64_t n = b->reader.unplaced.size(); for (auto& v : b->reader.by_tid) n += v.size(); return n; }
// host-side helpers of --partition-tag / --bedgraph, exposed for the CPU tests
int mkh_f32_display(float v, char* out, int cap) { const std::string s = f32_display(v); if ((int)s.size() + 1 > cap) return -1; memcpy(out, s.c_str(), s.size() + 1); return (int)s.size(); }
int mkh_pct2(float v, char* out, int cap) { char b[64]; char* e = put_pct2(b, v); const int n = (int)(e - b); if (n + 1 > cap) return -1; memcpy(out, b, n); out[n] = 0; return n; }
// partition key of the i-th record of tid (file order) for the ':'-separated tag list; returns 1 key, 0 NoKey, -1 error
int mkh_bam_partition_key(const mkh_bam* b, uint32_t tid, uint64_t i, const char* tags, char* out, int cap) {
    try {
        std::vector<std::string> tv;
        for (const char* p = tags; *p;) { const char* q = strchr(p, ':'); if (!q) q = p + strlen(p); tv.emplace_back(p, q - p); p = *q ? q + 1 : q; }
        const RecRef& r = b->reader.by_tid.at(tid).at(i);
        std::string k;
        const bool have = partition_key_of(b->reader.rec(r), r.size, tv, &k);
        if ((int)k.size() + 1 > cap) return -1;
        memcpy(out, k.c_str(), k.size() + 1);
        return have ? 1 : 0;
    } catch (const std::exception&) { return -1; }
}
// mapped-read count of a contig as the index-only open of the device front end sees it (BAI pseudo-bin; CPU only): -1 on error
int64_t mkh_bam_index_n_mapped(const char* bam_path, uint32_t tid) {
    try {
        BamReader bam;
        bam.open_device_index(bam_path, nullptr);
        if (!bam.have_index() || tid >= bam.stats.n_mapped.size()) return -1;
        return (int64_t)bam.stats.n_mapped[tid];
    } catch (const std::exception&) { return -1; }
}
// the key built from mkp_bam_tags cells (device front end): same return convention
int mkh_partition_key_of_cells(const uint8_t* cells, uint32_t n_tags, char* out, int cap) {
    std::string k;
    const bool have = partition_key_of_cells(cells, n_tags, &k);
    if ((int)k.size() + 1 > cap) return -1;
    memcpy(out, k.c_str(), k.size() + 1);
    return have ? 1 : 0;
}
void mkh_bam_close(mkh_bam* b) { delete b; }
uint32_t mkh_bam_n_refs(const mkh_bam* b) { return (uint32_t)b->reader.ref_names.size(); }
const char* mkh_bam_ref_name(const mkh_bam* b, uint32_t tid) { return b->reader.ref_names[tid].c_str(); }
uint32_t mkh_bam_ref_len(const mkh_bam* b, uint32_t tid) { return b->reader.ref_lens[tid]; }
uint64_t mkh_bam_n_mapped(const mkh_bam* b, uint32_t tid) { return b->reader.stats.n_mapped[tid]; }
uint64_t mkh_bam_n_records(const mkh_bam* b, uint32_t tid) { return b->reader.by_tid[tid].size(); }

int mkh_pack_region(const mkh_bam* b, uint32_t tid, uint32_t start, uint32_t end, mkh_packed** out) {
    try {
        mkh_packed* p = new mkh_packed();
        pack_region_mt(b->reader, tid, start, end, (int)std::min(32u, std::max(1u, std::thread::hardware_concurrency())), &p->pc);
        *out = p;
        return 0;
    }
    catch (const std::exception& e) { fprintf(stderr, "mkh_pack_region: %s\n", e.what()); return -1; }
}
void mkh_packed_free(mkh_packed* p) { delete p; }
uint32_t mkh_packed_n_reads(const mkh_packed* p) { return (uint32_t)p->pc.hdrs.size(); }
const mkp_read_hdr* mkh_packed_hdrs(const mkh_packed* p) { return p->pc.hdrs.data(); }
const uint8_t* mkh_packed_heap(const mkh_packed* p) { return p->pc.heap.data(); }
uint64_t mkh_packed_heap_bytes(const mkh_packed* p) { return p->pc.heap.size(); }
uint64_t mkh_packed_algorithmic_bytes(const mkh_packed* p) { return p->pc.algorithmic_bytes(); }

// bedMethyl text of device rows for an all-positions run (bench: rows -> text, writers.rs:87-156)
uint64_t mkh_format_rows(const mkp_row* rows, uint64_t n, const char* chrom, int mixed_delim, char* out, uint64_t cap) {
    BedFormat fmt; fmt.mixed_delim = mixed_delim != 0;
    std::string text;
    const std::string c = chrom;
    for (uint64_t i = 0; i < n; i++) { OutRow o{rows[i], -1, (char)rows[i].strand}; format_bed_row(o, c, fmt, &text); }
    if (out && text.size() <= cap) memcpy(out, text.data(), text.size());
    return text.size();
}

// Focus bitmaps (FocusPositions::check_position rules) of [start,end) for a motif list given as "CG:0,GATC:1".
// Intervals follow the reference grid (interval_size from `start`), so motif hits straddling an interval boundary are
// dropped exactly like the reference does (src/fasta.rs:207-227).
int mkh_motif_focus(const char* fasta, const char* contig, uint32_t start, uint32_t end, uint32_t interval_size,
                    const char* motifs, int combine_strands, uint32_t* pos_bits, uint32_t* neg_bits) {
    try {
        MotifContext mc;
        mc.fasta.open(fasta);
        std::string ms = motifs;
        for (size_t i = 0; i < ms.size();) {
            size_t j = ms.find(',', i); if (j == std::string::npos) j = ms.size();
            std::string one = ms.substr(i, j - i); size_t c = one.find(':');
            mc.motifs.push_back(parse_motif(one.substr(0, c), std::stoi(one.substr(c + 1))));
            mc.longest = std::max<uint64_t>(mc.longest, mc.motifs.back().len);
            i = j + 1;
        }
        std::vector<RefTarget> t{{0, start, end - start, contig}};
        std::vector<RefInterval> ivs = reference_intervals(t, interval_size, combine_strands != 0, &mc);
        std::vector<uint32_t> fp, fn;
        focus_bitmaps(ivs, 0, ivs.size(), start, end, &fp, &fn);
        memcpy(pos_bits, fp.data(), fp.size() * 4);
        memcpy(neg_bits, fn.data(), fn.size() * 4);
        return 0;
    } catch (const std::exception& e) { fprintf(stderr, "mkh_motif_focus: %s\n", e.what()); return -1; }
}

}  // extern "C"
