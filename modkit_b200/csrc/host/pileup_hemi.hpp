// `modkit pileup-hemi` orchestration on top of the device C ABI (mkp_hemi_resident). Mirrors DuplexModBamPileup::run
// (src/pileup/subcommand.rs:825-1514): one palindromic motif, intervals built with combine_strands = true, the threshold
// estimation of `modkit pileup`, rows written in feeder order by the hemi writer (src/writers.rs:185-255).
#pragma once
#include "pileup_run.hpp"

namespace mkh {

struct HemiOptions {
    PileupOptions p;            // the flags `pileup-hemi` shares with `pileup` (p.out_bed: -o, "" = stdout)
    bool have_seed = false;
};

// clap-compatible subset of the `modkit pileup-hemi` flag surface; every argument error is found here, before a device is opened
inline bool parse_hemi_args(int argc, const char* const* argv, HemiOptions* h, std::string* err) {
    PileupOptions* o = &h->p;
    std::vector<std::string> pos;
    for (int i = 0; i < argc; i++) {
        const std::string a = argv[i];
        auto val = [&]() -> std::string { if (i + 1 >= argc) throw std::runtime_error("a value is required for '" + a + "' but none was supplied"); return argv[++i]; };
        try {
            if (a == "-o" || a == "--out-bed") o->out_bed = val();
            else if (a == "-t" || a == "--threads") o->threads = std::stoi(val());
            else if (a == "-i" || a == "--interval-size") o->interval_size = (uint32_t)std::stoul(val());
            else if (a == "--region") o->region = val();
            else if (a == "--sample-region") o->sample_region = val();
            else if (a == "--sampling-interval-size") o->sampling_interval_size = (uint32_t)std::stoul(val());
            else if (a == "-n" || a == "--num-reads") o->num_reads = std::stoul(val());
            else if (a == "-f" || a == "--sampling-frac") { o->have_frac = true; o->frac = std::stod(val()); }
            else if (a == "--seed") { val(); h->have_seed = true; }
            else if (a == "--max-depth") o->max_depth = (uint32_t)std::stoul(val());
            else if (a == "--queue-size" || a == "--chunk-size" || a == "--log-filepath" || a == "--log") val();
            else if (a == "--no-filtering") o->no_filtering = true;
            else if (a == "-p" || a == "--filter-percentile") o->percentile = std::stof(val());
            else if (a == "--filter-threshold" || a == "--pass_threshold") o->filter_thresholds.push_back(val());
            else if (a == "--mod-thresholds" || a == "--mod-threshold") o->mod_thresholds.push_back(val());
            else if (a == "--include-unmapped") o->include_unmapped = true;
            else if (a == "--ignore") o->ignore = val();
            else if (a == "--force-allow-implicit") o->force_allow = true;
            else if (a == "--motif") { o->motif_parts.push_back(val()); o->motif_parts.push_back(val()); }
            else if (a == "--cpg") o->cpg = true;
            else if (a == "-r" || a == "--ref" || a == "--reference") o->ref_fp = val();
            else if (a == "-k" || a == "--mask") o->mask = true;
            else if (a == "--combine-mods") o->combine_mods = true;
            else if (a == "--edge-filter") o->edge = val();
            else if (a == "--invert-edge-filter") o->invert_edge = true;
            else if (a == "--only-tabs" || a == "--suppress-progress") {}
            else if (a == "--mixed-delim" || a == "--mixed-delimiters") o->mixed = true;
            else if (a == "--include-bed" || a == "--include-positions") o->include_bed = val();
            else if (a == "--device") o->device = std::stoi(val());
            else if (a == "--gpu-chunk-bp") o->chunk_bp = (uint32_t)std::stoul(val());
            else if (a == "--host-ingest") o->host_ingest = true;
            else if (a == "--quiet") o->quiet = true;
            else if (a == "--devices") { val(); *err = "pileup-hemi runs on one GPU: --devices is not supported (use --device N)"; return false; }
            else if (a.size() > 1 && a[0] == '-') { *err = "unexpected argument '" + a + "' found"; return false; }
            else pos.push_back(a);
        } catch (const std::exception& e) { *err = e.what(); return false; }
    }
    if (pos.size() != 1) { *err = "the following required arguments were not provided: <IN_BAM>"; return false; }
    o->in_bam = pos[0];
    if (o->ref_fp.empty()) { *err = "the following required arguments were not provided: --ref <REFERENCE_FASTA>"; return false; }
    if (o->cpg && !o->motif_parts.empty()) { *err = "the argument '--cpg' cannot be used with '--motif <MOTIF> <MOTIF>'"; return false; }
    if (o->combine_mods && !o->ignore.empty()) { *err = "the argument '--combine-mods' cannot be used with '--ignore <IGNORE>'"; return false; }
    const int n_thr = (o->no_filtering ? 1 : 0) + (o->filter_thresholds.empty() ? 0 : 1);
    if (n_thr > 1) { *err = "the argument '--no-filtering' cannot be used with '--filter-threshold <FILTER_THRESHOLD>'"; return false; }
    if (o->invert_edge && o->edge.empty()) { *err = "the following required arguments were not provided: --edge-filter <EDGE_FILTER>"; return false; }
    if (o->include_unmapped && !o->include_bed.empty()) { *err = "the argument '--include-unmapped' cannot be used with '--include-bed <INCLUDE_BED>'"; return false; }
    if (h->have_seed) { *err = "--seed selects Bernoulli read sampling (-f < 1.0), which is not reproducible here; use -n or -f 1.0"; return false; }
    if (o->have_frac && o->frac != 1.0) { *err = "only --sampling-frac 1.0 is reproducible without the reference's RNG; use -n or -f 1.0"; return false; }
    if (o->percentile > 1.0f) { *err = "filter percentile must be <= 1.0"; return false; }
    // the motif (subcommand.rs:1225-1262)
    if (!o->cpg) {
        if (o->motif_parts.empty()) { *err = "either --cpg or a --motif must be provided for pileup-hemi"; return false; }
        if (o->motif_parts.size() != 2) { *err = "motif arg should be length 2, eg. CG 0"; return false; }
        try { (void)std::stoul(o->motif_parts[1]); } catch (...) { *err = "couldn't parse focus position, " + o->motif_parts[1]; return false; }
    }
    try {
        const MotifSpec m = o->cpg ? parse_motif("CG", 0) : parse_motif(o->motif_parts[0], (int)std::stoul(o->motif_parts[1]));
        if (!m.palindromic) { *err = "motif must be palindromic for pileup-hemi"; return false; }
    } catch (const std::exception& e) { *err = e.what(); return false; }
    return true;
}

// one row of the hemi writer: chrom, pos, pos+1, "top,bottom,B", valid, '.', pos, pos+1, 255,0,0, valid, pct, count, n_canonical,
// n_other_pattern, n_delete, n_fail, n_diff, n_nocall; the columns after the tenth are separated by spaces with --mixed-delim
inline void format_hemi_row(const mkp_hemi_row& r, const std::string& chrom, bool mixed, std::string* out) {
    const char sp = mixed ? ' ' : '\t';
    const uint32_t valid = r.count + r.n_other_pattern;
    char buf[512];
    char* p = buf;
    auto half = [&](uint32_t code) {
        if (code == 0) *p++ = '-';
        else if (code & 0x80000000u) p = put_u32(p, code & 0x7fffffffu);
        else *p++ = (char)code;
    };
    out->append(chrom);
    *p++ = '\t'; p = put_u32(p, r.pos); *p++ = '\t'; p = put_u32(p, r.pos + 1); *p++ = '\t';
    half(r.top_code); *p++ = ','; half(r.bottom_code); *p++ = ','; *p++ = "ACGT"[r.primary_base & 3];
    *p++ = '\t'; p = put_u32(p, valid); memcpy(p, "\t.\t", 3); p += 3; p = put_u32(p, r.pos); *p++ = '\t'; p = put_u32(p, r.pos + 1);
    memcpy(p, "\t255,0,0\t", 9); p += 9;
    p = put_u32(p, valid); *p++ = sp;
    const float frac = (float)r.count / (float)valid;        // frac_pattern() * 100f32, printed with {:.2}
    volatile float pct = frac * 100.0f;
    p = put_pct2(p, pct);
    *p++ = sp; p = put_u32(p, r.count); *p++ = sp; p = put_u32(p, r.n_canonical); *p++ = sp; p = put_u32(p, r.n_other_pattern);
    *p++ = sp; p = put_u32(p, r.n_delete); *p++ = sp; p = put_u32(p, r.n_fail); *p++ = sp; p = put_u32(p, r.n_diff);
    *p++ = sp; p = put_u32(p, r.n_nocall); *p++ = '\n';
    out->append(buf, (size_t)(p - buf));
}

inline int run_pileup_hemi(const HemiOptions& h, RunSummary* summary, std::string* error) {
    using clk = std::chrono::steady_clock;
    auto secs = [](clk::time_point a, clk::time_point b) { return std::chrono::duration<double>(b - a).count(); };
    const PileupOptions& o = h.p;
    try {
        const auto t0 = clk::now();
        DeviceGuard dev;
        {
            const int rc = mkp_create(o.device, &dev.ctx);
            if (rc) throw std::runtime_error("no usable CUDA device (mkp_create returned " + std::to_string(rc) + "); this build has no CPU fallback");
        }
        BamReader bam;
        if (o.host_ingest) bam.open(o.in_bam, o.threads);
        else bam.open_device_index(o.in_bam, dev.ctx);
        Region region, sregion;
        const Region* rp = nullptr; const Region* srp = nullptr;
        if (!o.region.empty()) { region = parse_region_arg(o.region, bam); rp = &region; }
        if (!o.sample_region.empty()) { sregion = parse_region_arg(o.sample_region, bam); srp = &sregion; }
        std::vector<RefTarget> targets;
        for (uint32_t t = 0; t < bam.ref_names.size(); t++) {
            if (rp) { if (bam.ref_names[t] == rp->name) targets.push_back({t, rp->start, rp->end - rp->start, rp->name}); }
            else targets.push_back({t, 0, bam.ref_lens[t], bam.ref_names[t]});
        }
        IncludeBed include;
        const IncludeBed* inc = nullptr;
        if (!o.include_bed.empty()) {
            std::map<std::string, uint32_t> name_to_tid;
            for (auto& t : targets) name_to_tid[t.name] = t.tid;
            include.read(o.include_bed, name_to_tid);
            inc = &include;
        }
        mkp_params P;
        memset(&P, 0, sizeof P);
        P.force_allow_implicit = o.force_allow;
        P.max_depth = o.max_depth;
        if (o.combine_mods) P.numeric_mode = 1;
        else if (!o.ignore.empty()) { uint32_t c; if (!parse_code(o.ignore, &c)) throw std::runtime_error("failed to parse mod code " + o.ignore); P.numeric_mode = 2; P.collapse_code = c; }
        if (!o.edge.empty()) {
            P.edge_filter_on = 1; P.edge_filter_inverted = o.invert_edge;
            auto c = o.edge.find(',');
            if (c == std::string::npos) P.edge_filter_start = P.edge_filter_end = (uint32_t)std::stoul(o.edge);
            else { P.edge_filter_start = (uint32_t)std::stoul(o.edge.substr(0, c)); P.edge_filter_end = (uint32_t)std::stoul(o.edge.substr(c + 1)); }
        }
        MotifContext mc;
        mc.motifs.push_back(o.cpg ? parse_motif("CG", 0) : parse_motif(o.motif_parts[0], (int)std::stoul(o.motif_parts[1])));
        const MotifSpec& motif = mc.motifs[0];
        const int32_t offset = motif.rc_offset - motif.offset;     // MotifInfo::offset (motif_bed.rs:111-141)
        mc.fasta.open(o.ref_fp);
        mc.keep_case = o.mask;
        mc.include = inc;
        mc.longest = (uint64_t)motif.len;
        std::vector<RefTarget> iv_targets = targets;
        if (inc) iv_targets = targets_from_include_bed(*inc, iv_targets, o.interval_size);
        std::vector<size_t> iv_owner;
        std::vector<RefInterval> ivs = interval_grid(iv_targets, o.interval_size, true, &mc, &iv_owner);   // combine_strands = true (:1383-1390)
        fill_interval_focus(ivs, 0, ivs.size(), iv_targets, iv_owner, true, &mc, inc, std::max(1, o.threads / 2));
        if (!o.host_ingest) {
            try { bam.load_default(); }
            catch (const DeviceIngestTooBig& e) {
                if (!o.quiet) fprintf(stderr, "> %s; reading the BAM on the host instead\n", e.what());
                bam = BamReader();
                bam.open(o.in_bam, o.threads);
            }
        }
        const auto t_load = clk::now();
        uint64_t any_mapped = 0;
        for (auto& t : targets) if (rp || !inc || inc->has_contig(t.tid)) any_mapped += bam.stats.n_mapped[t.tid];
        if (!any_mapped) throw std::runtime_error("did not find any mapped reads, perform alignment first or use modkit extract and/or modkit summary to inspect unaligned modBAMs");
        FILE* out = o.out_bed.empty() || o.out_bed == "-" ? stdout : fopen(o.out_bed.c_str(), "w");
        if (!out) throw std::runtime_error("failed to make output file");
        struct Closer { FILE* f; ~Closer() { if (f && f != stdout) fclose(f); } } closer{out};

        // thresholds: the same estimation as `modkit pileup` (get_threshold_from_options)
        for (auto& raw : o.mod_thresholds) {
            auto c = raw.find(':');
            uint32_t code;
            if (c == std::string::npos || raw.find(':', c + 1) != std::string::npos || !parse_code(raw.substr(0, c), &code))
                throw std::runtime_error("encountered illegal per-mod threshold: " + raw + ". Should be mod_code:threshold e.g. h:0.8");
            if (P.n_mod_thresholds >= MKP_MAX_MOD_THRESHOLDS) throw std::runtime_error("too many per-mod thresholds");
            P.mod_code[P.n_mod_thresholds] = code;
            P.mod_threshold[P.n_mod_thresholds++] = std::stof(raw.substr(c + 1));
        }
        if (!o.filter_thresholds.empty()) {
            bool have_default = false;
            for (auto& raw : o.filter_thresholds) {
                auto c = raw.find(':');
                if (c == std::string::npos) {
                    if (have_default) throw std::runtime_error("default threshold encountered more than once");
                    P.default_threshold = std::stof(raw); have_default = true;
                } else {
                    const char* B = "ACGT";
                    const char* f = raw.empty() ? nullptr : strchr(B, raw[0]);
                    if (!f || !raw[0]) throw std::runtime_error("failed to parse base " + raw);
                    if (P.base_threshold_set[f - B]) throw std::runtime_error(std::string("repeated threshold for base ") + raw[0]);
                    P.base_threshold_set[f - B] = 1;
                    P.base_threshold[f - B] = std::stof(raw.substr(c + 1));
                }
            }
        } else if (!o.no_filtering) {
            mkp_params PS = P;
            PS.max_depth = 0;
            if (mkp_set_params(dev.ctx, &PS)) throw std::runtime_error(mkp_last_error(dev.ctx));
            SamplerConfig sc;
            sc.threads = o.threads; sc.workers = o.threads; sc.sampling_interval_size = o.sampling_interval_size;
            sc.take_all = o.have_frac;
            sc.num_reads = o.num_reads;
            sc.region = srp ? srp : rp;
            sc.include_unmapped = o.include_unmapped;
            sc.edge_on = P.edge_filter_on;
            sc.include = inc;
            std::vector<uint64_t> hist(4 * 1025);
            uint64_t inexact = 0;
            double fetch_s = 0;
            if (bam.on_device && bam.have_index()) sample_histogram_indexed(bam, dev.ctx, sc, hist.data(), &inexact, Collective(), &fetch_s);
            else sample_histogram(bam, dev.ctx, sc, hist.data(), &inexact);
            if (inexact) throw std::runtime_error("sampled probabilities are not multiples of 1/1024 (" + std::to_string(inexact) + " values): exact histogram quantile impossible; pass --filter-threshold");
            for (int b = 0; b < 4; b++) {
                float thr;
                uint64_t n = 0;
                for (int k = 0; k <= 1024; k++) n += hist[b * 1025 + k];
                if (!n) continue;
                if (!percentile_from_hist(hist.data() + b * 1025, o.percentile, &thr)) throw std::runtime_error("not enough datapoints to estimate a threshold");
                P.base_threshold_set[b] = 1;
                P.base_threshold[b] = thr;
                if (!o.quiet) fprintf(stderr, "> Using filter threshold %.9g for %c.\n", thr, "ACGT"[b]);
            }
        }
        if (mkp_set_params(dev.ctx, &P)) throw std::runtime_error(mkp_last_error(dev.ctx));
        const auto t_thr = clk::now();

        // chunks: consecutive intervals of one contig up to --gpu-chunk-bp. k_resolve keeps the calls inside the chunk range only,
        // so the range reaches |offset| past the columns on the partner's side: every partner has its call records.
        RunSummary S;
        for (auto& iv : ivs) S.positions += iv.end - iv.start;
        const uint32_t pad_lo = offset < 0 ? (uint32_t)-offset : 0u, pad_hi = offset > 0 ? (uint32_t)offset : 0u;
        PackedChunk pc;
        std::vector<uint32_t> fpos, fneg, cols, partners, starts;
        std::string text;
        for (size_t c0 = 0; c0 < ivs.size();) {
            size_t c1 = c0 + 1;
            while (c1 < ivs.size() && ivs[c1].tid == ivs[c0].tid && ivs[c1].start == ivs[c1 - 1].end && ivs[c1].end - ivs[c0].start <= o.chunk_bp) c1++;
            if (ivs[c1 - 1].end <= ivs[c0].start) { c0 = c1; continue; }
            std::vector<RecRef> chunk_recs;
            bam.ensure_tid(ivs[c0].tid);
            bam.for_overlapping(ivs[c0].tid, ivs[c0].start, ivs[c1 - 1].end, [&](const RecRef& r) { chunk_recs.push_back(r); });
            if (chunk_recs.empty()) { c0 = c1; continue; }
            // --max-depth: htslib's engine runs per interval (as for `modkit pileup`, depth_limit_keep)
            struct Work { size_t a, b; std::vector<RecRef> recs; };
            std::vector<Work> work;
            bool split = false;
            if (o.max_depth && chunk_recs.size() > o.max_depth) {
                std::vector<Work> per_iv;
                for (size_t k = c0; k < c1; k++) {
                    Work w{k, k + 1, {}};
                    for (auto& r : chunk_recs) if (r.pos < (int64_t)ivs[k].end && r.end > (int64_t)ivs[k].start) w.recs.push_back(r);
                    const size_t before = w.recs.size();
                    depth_limit_keep(&w.recs, o.max_depth);
                    split = split || w.recs.size() != before;
                    per_iv.push_back(std::move(w));
                }
                if (split) work.swap(per_iv);
            }
            if (!split) { Work w{c0, c1, {}}; w.recs.swap(chunk_recs); work.push_back(std::move(w)); }
            for (auto& wk : work) {
                const size_t i0 = wk.a, i1 = wk.b;
                const uint32_t a = ivs[i0].start, b = ivs[i1 - 1].end;
                if (b <= a || wk.recs.empty()) continue;
                const uint32_t cs = a > pad_lo ? a - pad_lo : 0u, ce = b + pad_hi;
                // columns = the '+' motif positions (positive_motifs of FocusPositions::MotifCombineStrands); partners = column + offset
                focus_bitmaps(ivs, i0, i1, cs, ce, &fpos, &fneg);
                cols.assign(fpos.size(), 0); partners.assign(fpos.size(), 0);
                size_t n_cols = 0;
                for (size_t w = 0; w < fpos.size(); w++) for (uint32_t bits = fpos[w]; bits; bits &= bits - 1) {
                    const uint32_t x = (uint32_t)(w * 32 + __builtin_ctz(bits)), p = cs + x;
                    if (p < a || p >= b) continue;
                    const int64_t q = (int64_t)p + offset;
                    cols[w] |= 1u << (x & 31);
                    n_cols++;
                    if (q >= (int64_t)cs && q < (int64_t)ce) { const uint32_t y = (uint32_t)(q - cs); partners[y >> 5] |= 1u << (y & 31); }
                }
                if (!n_cols) continue;
                starts.clear();
                for (size_t i = i0; i < i1; i++) starts.push_back(ivs[i].start);
                pc.clear();
                if (bam.on_device) pc.recs = wk.recs;
                else pack_records_mt(bam, wk.recs, o.threads, &pc);
                if (pc.recs.empty()) continue;
                mkp_stats st;
                if (bam.on_device) device_chunk(bam, pc.recs, cs, ce, cols.data(), partners.data());
                else {
                    mkp_chunk ch;
                    memset(&ch, 0, sizeof ch);
                    ch.start = cs; ch.end = ce; ch.hdrs = pc.hdrs.data(); ch.n_reads = (uint32_t)pc.hdrs.size(); ch.heap = pc.heap.data(); ch.heap_bytes = pc.heap.size();
                    ch.focus_pos = cols.data(); ch.focus_neg = partners.data();
                    if (mkp_upload_chunk(dev.ctx, &ch)) throw std::runtime_error(mkp_last_error(dev.ctx));
                }
                if (mkp_hemi_resident(dev.ctx, offset, starts.data(), (uint32_t)starts.size(), &st)) throw std::runtime_error(mkp_last_error(dev.ctx));
                const mkp_hemi_row* rows = nullptr;
                size_t n_rows = 0;
                if (mkp_fetch_hemi_rows(dev.ctx, &rows, &n_rows)) throw std::runtime_error(mkp_last_error(dev.ctx));
                const std::string& chrom = bam.ref_names[ivs[i0].tid];
                text.clear();
                for (size_t k = 0; k < n_rows; k++) format_hemi_row(rows[k], chrom, o.mixed, &text);
                if (!text.empty() && fwrite(text.data(), 1, text.size(), out) != text.size()) throw std::runtime_error("failed to write output file " + o.out_bed);
                S.rows += n_rows;
                S.kernel_ms += st.kernel_ms[7];
                S.reads_packed += pc.recs.size();
                S.chunks++;
            }
            c0 = c1;
        }
        fflush(out);
        const auto t1 = clk::now();
        S.load_s = secs(t0, t_load); S.threshold_s = secs(t_load, t_thr); S.total_s = secs(t0, t1); S.rows_total = S.rows; S.positions_total = S.positions;
        for (int b = 0; b < 4; b++) { S.thresholds[b] = P.base_threshold[b]; S.threshold_set[b] = P.base_threshold_set[b]; }
        if (summary) *summary = S;
        if (!o.quiet)
            fprintf(stderr, "> Done, processed %llu rows. positions=%llu reads=%llu chunks=%llu (kernels %.3f ms) total=%.3fs\n",
                    (unsigned long long)S.rows, (unsigned long long)S.positions, (unsigned long long)S.reads_packed, (unsigned long long)S.chunks, S.kernel_ms, S.total_s);
        return 0;
    } catch (const std::exception& e) {
        if (error) *error = e.what();
        return 1;
    }
}

}  // namespace mkh
