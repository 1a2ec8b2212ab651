// CHECKER — TEST INFRASTRUCTURE ONLY. Never linked into or called from the product path.
//
// `hemi_oracle [flags] <in.bam> [-o out.bed]`: CPU restatement of `modkit pileup-hemi` (reference v0.4.4) on top of the
// pileup oracle's BAM reader, MM/ML decode, threshold caller, interval feeder and motif search (oracle/*.hpp, used as they
// are). It walks every interval column by column the way htslib's pileup engine hands them to the reference, so the
// per-interval read cache and its skip set behave as they do there.
//   flags and run            src/pileup/subcommand.rs:825-1514 (DuplexModBamPileup)
//   per-interval loop        src/pileup/duplex.rs:238-339 (process_region_duplex)
//   counts -> rows           src/pileup/duplex.rs:84-205 (DuplexFeatureVector::decode)
//   read cache               src/read_cache.rs:111-297 (ReadCache::add_record / get_mod_call), 368-463 (DuplexReadCache)
//   call pairs               src/mod_bam.rs:1674-1830 (DuplexModCall, DuplexModCodeRepr)
//   row text                 src/writers.rs:185-255
#include <atomic>
#include <condition_variable>

#include "../oracle/driver.hpp"

using namespace orc;

static void die(const std::string& m) { fprintf(stderr, "> Error! %s\n", m.c_str()); exit(1); }

// one read of the per-interval cache: its calls by (mod strand, MM base) and reference position, or skipped
struct HemiRead {
    bool decoded = false, skipped = false;
    std::map<uint32_t, Call> tab[2][4];
};

// ReadCache::add_record: false = the read goes to the skip set
static bool decode_hemi_read(const BamRecord& r, const PileupParams& P, HemiRead* out) {
    ModBaseInfo info;
    std::string fwd;
    if (!decode_mod_base_info(r, &info, &fwd) || info.is_empty()) return false;
    for (int s = 0; s < 2; s++) for (int b = 0; b < 4; b++)
        if (info.present[s][b] && info.tab[s][b].mode == DEFAULT_IMPLICIT && !P.force_allow_implicit) return false;
    const int L = r.l_seq();
    const bool rev = r.is_reverse();
    std::vector<int64_t> q2r;
    aligned_ref_positions(r, &q2r);
    bool added = false;
    for (int s = 0; s < 2; s++) for (int b = 0; b < 4; b++) {
        if (!info.present[s][b]) continue;
        SeqPosTable& T = info.tab[s][b];
        if (P.edge.on) {
            if (!P.edge.read_can_be_trimmed((size_t)L)) continue;
            for (auto it = T.pos.begin(); it != T.pos.end();) { if (!P.edge.keep(it->first, (size_t)L)) it = T.pos.erase(it); else ++it; }
            if (T.pos.empty()) continue;
        }
        const int tb = s == 0 ? b : comp_idx(b);          // the base the modification is called on
        for (auto& kv : T.pos) {
            const int q = rev ? L - 1 - (int)kv.first : (int)kv.first;
            if (q < 0 || q >= L || q2r[q] < 0) continue;
            const BaseModProbs bmp = P.numeric == COLLAPSE ? redistribute(kv.second, P.collapse_code) : kv.second;
            out->tab[s][b][(uint32_t)q2r[q]] = make_call(P.caller, tb, bmp);
        }
        added = true;
    }
    return added;
}

// DuplexModCodeRepr in its derived order: Canonical < Code(char) < ChEbi(n)
static uint64_t half_key(const Call& c) { return c.kind == CALL_CANONICAL ? 0 : (c.code & 0x80000000u) ? (1ull << 32) + (c.code & 0x7fffffffu) : 1ull + c.code; }
static std::string half_text(uint64_t k) { return k == 0 ? std::string("-") : k > (1ull << 32) ? std::to_string(k - (1ull << 32)) : std::string(1, (char)(k - 1)); }

struct HemiColumn {
    uint32_t n_delete = 0;
    std::map<std::pair<uint64_t, uint64_t>, uint32_t> patterns[4];   // per primary (read) base
    uint32_t n_fail[4] = {0, 0, 0, 0}, n_nocall[4] = {0, 0, 0, 0};
};

static void process_interval_hemi(const BamFile& bam, const Interval& iv, const PileupParams& P, int offset, const std::string& chrom,
                                  bool mixed, std::string* text, size_t* n_rows) {
    if (iv.end <= iv.start) return;
    std::vector<uint32_t> cols;
    for (auto& kv : iv.focus.pos_ids) if (kv.first >= iv.start && kv.first < iv.end && !kv.second.empty()) cols.push_back(kv.first);
    if (cols.empty()) return;
    std::vector<const BamRecord*> recs;
    {
        std::vector<const BamRecord*> pushed;
        bam.fetch(iv.tid, iv.start, iv.end, [&](const BamRecord& r) { if (!(r.flag() & (0x4 | 0x100 | 0x200 | 0x400))) pushed.push_back(&r); });
        plp_maxcnt_filter(&pushed, P.max_depth);
        for (const BamRecord* r : pushed) if (admitted_for_pileup(*r)) recs.push_back(r);
    }
    if (recs.empty()) return;
    // per read: CIGAR ops with reference length as (ref start, op, len, query start)
    struct Op { int64_t r0; int op; int len; int q0; };
    std::vector<std::vector<Op>> ops(recs.size());
    std::vector<int64_t> rend(recs.size());
    for (size_t i = 0; i < recs.size(); i++) {
        const BamRecord& r = *recs[i];
        int64_t rp = r.pos();
        int q = 0;
        for (int ci = 0; ci < r.n_cigar(); ci++) {
            const uint32_t c = r.cigar_op(ci);
            const int op = c & 0xf, len = (int)(c >> 4);
            if (op == 0 || op == 7 || op == 8) { ops[i].push_back({rp, op, len, q}); rp += len; q += len; }
            else if (op == 1 || op == 4) q += len;
            else if (op == 2 || op == 3) { ops[i].push_back({rp, op, len, q}); rp += len; }
        }
        rend[i] = rp;
    }
    std::vector<HemiRead> cache(recs.size());              // one read cache per interval (duplex.rs:266-271)
    for (uint32_t p : cols) {
        HemiColumn C;
        bool any = false;
        for (size_t i = 0; i < recs.size(); i++) {
            const BamRecord& r = *recs[i];
            if ((int64_t)p < r.pos() || (int64_t)p >= rend[i]) continue;
            const auto& ov = ops[i];
            size_t k = std::upper_bound(ov.begin(), ov.end(), (int64_t)p, [](int64_t x, const Op& o) { return x < o.r0; }) - ov.begin();
            if (k == 0) continue;
            const Op& o = ov[k - 1];
            if ((int64_t)p >= o.r0 + o.len) continue;
            any = true;
            if (o.op == 3) continue;                          // reference skip: not part of the column
            if (o.op == 2) { C.n_delete++; continue; }        // counted before any read-cache lookup
            const int q = o.q0 + (int)(p - o.r0);
            if (q >= r.l_seq()) continue;
            const int b = base_idx(r.base_at(q));             // the stored base (reference orientation)
            if (b < 0) continue;
            HemiRead& H = cache[i];
            if (H.skipped) continue;
            if (!H.decoded) {                                 // first lookup: add_record, or the skip set and one NoCall
                H.decoded = true;
                if (!decode_hemi_read(r, P, &H)) { H.skipped = true; C.n_nocall[b]++; continue; }
            }
            const bool rev = r.is_reverse();
            const int cb = comp_idx(b);
            const std::map<uint32_t, Call>& top = rev ? H.tab[1][cb] : H.tab[0][b];
            const std::map<uint32_t, Call>& bot = rev ? H.tab[0][b] : H.tab[1][cb];
            const int64_t partner = (int64_t)p + offset;
            auto t = top.find(p);
            auto u = partner >= 0 ? bot.find((uint32_t)partner) : bot.end();
            if (t == top.end() || u == bot.end()) { C.n_nocall[b]++; continue; }
            if (t->second.kind == CALL_FILTERED || u->second.kind == CALL_FILTERED) { C.n_fail[b]++; continue; }
            uint64_t k0 = half_key(t->second), k1 = half_key(u->second);
            if (P.numeric == COMBINE) { if (k0) k0 = 1ull + (uint8_t)BASES[b]; if (k1) k1 = 1ull + (uint8_t)BASES[b]; }
            C.patterns[b][{k0, k1}]++;
        }
        if (!any) continue;
        uint32_t mod_calls[4] = {0, 0, 0, 0};
        for (int b = 0; b < 4; b++) for (auto& kv : C.patterns[b]) mod_calls[b] += kv.second;
        const char sp = mixed ? ' ' : '\t';
        for (int b = 0; b < 4; b++) {
            if (C.patterns[b].empty()) continue;
            uint32_t n_diff = 0;
            for (int o = 0; o < 4; o++) if (o != b) n_diff += mod_calls[o];
            auto cz = C.patterns[b].find({0, 0});
            const uint32_t n_canon = cz == C.patterns[b].end() ? 0 : cz->second;
            for (auto& kv : C.patterns[b]) {
                const uint32_t count = kv.second, other = mod_calls[b] - count, valid = count + other;
                volatile float frac = (float)count / (float)valid;
                volatile float pct = frac * 100.0f;
                char buf[512];
                const std::string name = half_text(kv.first.first) + "," + half_text(kv.first.second) + "," + BASES[b];
                const int n = snprintf(buf, sizeof buf, "%s\t%u\t%u\t%s\t%u\t.\t%u\t%u\t255,0,0\t%u%c%.2f%c%u%c%u%c%u%c%u%c%u%c%u%c%u\n",
                                       chrom.c_str(), p, p + 1, name.c_str(), valid, p, p + 1, valid, sp, (double)pct, sp, count, sp, n_canon,
                                       sp, other, sp, C.n_delete, sp, C.n_fail[b], sp, n_diff, sp, C.n_nocall[b]);
                text->append(buf, (size_t)n);
                (*n_rows)++;
            }
        }
    }
}

int main(int argc, char** argv) {
    try {
        std::vector<std::string> pos;
        int threads = 4;
        uint32_t interval_size = 100000, sampling_interval_size = 1000000, max_depth = 8000;
        size_t num_reads = 10042;
        bool have_frac = false, no_filtering = false, include_unmapped = false, force_allow = false, cpg = false, mask = false;
        bool combine_mods = false, mixed = false, invert_edge = false;
        double frac = 0;
        float percentile = 0.1f;
        std::vector<std::string> filter_thresholds, mod_thresholds, motif_parts;
        std::string region_s, sample_region_s, ignore_s, ref_fp, edge_s, include_bed, out_fp;
        for (int i = 1; i < argc; i++) {
            std::string a = argv[i];
            auto val = [&]() -> std::string { if (i + 1 >= argc) die("missing value for " + a); return argv[++i]; };
            if (a == "-t" || a == "--threads") threads = std::stoi(val());
            else if (a == "-o" || a == "--out-bed") out_fp = val();
            else if (a == "-i" || a == "--interval-size") interval_size = (uint32_t)std::stoul(val());
            else if (a == "--region") region_s = val();
            else if (a == "--sample-region") sample_region_s = val();
            else if (a == "--sampling-interval-size") sampling_interval_size = (uint32_t)std::stoul(val());
            else if (a == "-n" || a == "--num-reads") num_reads = std::stoul(val());
            else if (a == "-f" || a == "--sampling-frac") { have_frac = true; frac = std::stod(val()); }
            else if (a == "--max-depth") max_depth = (uint32_t)std::stoul(val());
            else if (a == "--queue-size" || a == "--chunk-size" || a == "--log-filepath" || a == "--log") val();
            else if (a == "--no-filtering") no_filtering = true;
            else if (a == "-p" || a == "--filter-percentile") percentile = std::stof(val());
            else if (a == "--filter-threshold" || a == "--pass_threshold") filter_thresholds.push_back(val());
            else if (a == "--mod-thresholds" || a == "--mod-threshold") mod_thresholds.push_back(val());
            else if (a == "--include-unmapped") include_unmapped = true;
            else if (a == "--ignore") ignore_s = val();
            else if (a == "--force-allow-implicit") force_allow = true;
            else if (a == "--motif") { motif_parts.push_back(val()); motif_parts.push_back(val()); }
            else if (a == "--cpg") cpg = true;
            else if (a == "-r" || a == "--ref" || a == "--reference") ref_fp = val();
            else if (a == "-k" || a == "--mask") mask = true;
            else if (a == "--combine-mods") combine_mods = true;
            else if (a == "--edge-filter") edge_s = val();
            else if (a == "--invert-edge-filter") invert_edge = true;
            else if (a == "--only-tabs" || a == "--suppress-progress") {}
            else if (a == "--mixed-delim" || a == "--mixed-delimiters") mixed = true;
            else if (a == "--include-bed" || a == "--include-positions") include_bed = val();
            else if (a.size() > 1 && a[0] == '-') die("unsupported flag " + a);
            else pos.push_back(a);
        }
        if (pos.size() != 1) die("usage: hemi_oracle [flags] <in.bam> [-o out.bed]");
        if (cpg && !motif_parts.empty()) die("the argument '--cpg' cannot be used with '--motif <MOTIF> <MOTIF>'");
        if (ref_fp.empty()) die("the following required arguments were not provided: --ref <REFERENCE_FASTA>");
        BamFile bam;
        bam.load(pos[0], threads);
        Region region, sample_region;
        const Region* rp = nullptr; const Region* srp = nullptr;
        if (!region_s.empty()) { region = parse_region(region_s, bam); rp = &region; }
        if (!sample_region_s.empty()) { sample_region = parse_region(sample_region_s, bam); srp = &sample_region; }
        std::vector<RefRecord> targets = get_targets(bam, rp);
        PositionFilter pfilter;
        const PositionFilter* pf = nullptr;
        if (!include_bed.empty()) {
            std::map<std::string, uint32_t> c2t;
            for (auto& t : targets) c2t[t.name] = t.tid;
            pfilter.load(include_bed, c2t);
            pf = &pfilter;
        }
        {
            uint64_t mapped = 0;
            for (auto& t : targets) if (rp || !pf || pf->has_contig(t.tid)) mapped += bam.n_mapped[t.tid];
            if (!mapped) die("did not find any mapped reads, perform alignment first or use modkit extract and/or modkit summary to inspect unaligned modBAMs");
        }
        if (percentile > 1.0f) die("filter percentile must be <= 1.0");
        PileupParams P;
        P.max_depth = max_depth;
        P.force_allow_implicit = force_allow;
        bool threshold_collapse = false;
        if (combine_mods) P.numeric = COMBINE;
        else if (!ignore_s.empty()) {
            ModCode c;
            if (!parse_mod_code(ignore_s, &c)) die("failed to parse mod code " + ignore_s);
            P.numeric = COLLAPSE; P.collapse_code = c; threshold_collapse = true;
        }
        P.combine_strands = true;
        if (!edge_s.empty()) {
            P.edge.on = true; P.edge.inverted = invert_edge;
            auto c = edge_s.find(',');
            if (c == std::string::npos) P.edge.start = P.edge.end = std::stoul(edge_s);
            else { P.edge.start = std::stoul(edge_s.substr(0, c)); P.edge.end = std::stoul(edge_s.substr(c + 1)); }
        }
        Motif motif;
        if (cpg) motif = Motif::parse("CG", 0);
        else {
            if (motif_parts.empty()) die("either --cpg or a --motif must be provided for pileup-hemi");
            if (motif_parts.size() != 2) die("motif arg should be length 2, eg. CG 0");
            motif = Motif::parse(motif_parts[0], std::stoi(motif_parts[1]));
        }
        if (!motif.palindrome) die("motif must be palindromic for pileup-hemi");
        const int offset = motif.rev_off - motif.fwd_off;   // MotifInfo::offset (motif_bed.rs:111-141)
        std::vector<Motif> motifs{motif};
        MotifLookup lookup;
        lookup.fa.open(ref_fp);
        lookup.motifs = motifs;
        lookup.mask = mask;
        lookup.pf = pf;
        lookup.longest = motif.length;
        for (auto& raw : mod_thresholds) {
            auto c = raw.find(':');
            ModCode code;
            if (c == std::string::npos || !parse_mod_code(raw.substr(0, c), &code)) die("illegal per-mod threshold " + raw);
            P.caller.mod_thr.push_back({code, std::stof(raw.substr(c + 1))});
        }
        if (!filter_thresholds.empty()) {
            for (auto& raw : filter_thresholds) {
                auto c = raw.find(':');
                if (c == std::string::npos) { P.caller.default_thr = std::stof(raw); continue; }
                const int b = base_idx(raw[0]);
                if (b < 0) die("failed to parse base " + raw);
                P.caller.base_set[b] = true;
                P.caller.base_thr[b] = std::stof(raw.substr(c + 1));
            }
        } else if (!no_filtering) {
            SampleOptions so;
            so.threads = threads;
            so.sampling_interval_size = sampling_interval_size;
            if (have_frac) { if (frac != 1.0) die("only -f 1.0 is supported"); so.frac_all = true; }
            so.num_reads = num_reads;
            so.region = srp ? srp : rp;
            so.include_unmapped = include_unmapped;
            so.collapse = threshold_collapse;
            so.collapse_code = P.collapse_code;
            so.edge = P.edge;
            so.pf = pf;
            estimate_thresholds(bam, so, percentile, &P.caller);
            for (int b = 0; b < 4; b++) if (P.caller.base_set[b]) fprintf(stderr, "> Using filter threshold %.9g for %c.\n", P.caller.base_thr[b], BASES[b]);
        }
        if (pf) targets = optimize_reference_records(*pf, targets, interval_size);
        std::vector<Interval> ivs = make_intervals(targets, interval_size, true, &lookup, nullptr, pf);
        FILE* out = out_fp.empty() ? stdout : fopen(out_fp.c_str(), "w");
        if (!out) die("failed to make output file");
        std::vector<std::string> results(ivs.size());
        std::vector<char> done(ivs.size(), 0);
        std::atomic<size_t> next{0};
        std::mutex mu;
        std::condition_variable cv;
        size_t n_rows = 0;
        auto worker = [&]() {
            for (;;) {
                const size_t i = next.fetch_add(1);
                if (i >= ivs.size()) break;
                std::string text;
                size_t nr = 0;
                process_interval_hemi(bam, ivs[i], P, offset, bam.ref_names[ivs[i].tid], mixed, &text, &nr);
                std::lock_guard<std::mutex> g(mu);
                results[i].swap(text);
                done[i] = 1;
                n_rows += nr;
                cv.notify_all();
            }
        };
        std::vector<std::thread> pool;
        for (int t = 0; t < std::max(1, threads); t++) pool.emplace_back(worker);
        for (size_t i = 0; i < ivs.size(); i++) {
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return done[i] != 0; });
            std::string text;
            text.swap(results[i]);
            lk.unlock();
            fwrite(text.data(), 1, text.size(), out);
        }
        for (auto& t : pool) t.join();
        if (out != stdout) fclose(out); else fflush(out);
        fprintf(stderr, "> Done, processed %zu rows.\n", n_rows);
        return 0;
    } catch (const std::exception& e) {
        die(e.what());
    }
    return 1;
}
