// Deterministic synthetic modBAM generator (SURVEY.md Appendix D): reference FASTA (+.fai) and a
// coordinate-sorted BAM (+.bai) of ONT-like reads carrying MM/ML base-modification tags.
// Test / bench infrastructure: produces the SAME file for the CPU oracle, the GPU product and (if one is
// ever available) the real `modkit` binary.
//
//   synth_modbam --out PREFIX [--contig NAME:LEN]... [--coverage 30] [--seed 20260924] [--mods m|hm|hma]
//                [--mean-len 12000] [--level 1] [--threads 8] [--combined-hm] [--implicit] [--odd-records] [--partition-tags [--long-rg]]
//                [--start-grid G]  (read starts snapped to multiples of G: stacks of reads sharing a start, for --max-depth)
//                [--region-only START-END]   (only reads overlapping the window; reference still full length)
//                [--duplex]  (each read also carries G-h?/G-m? lists: calls on the opposite strand's C of every CpG, drawn
//                             independently, so hemi-methylated patterns occur; `modkit pileup-hemi` input)
// Writes PREFIX.fa, PREFIX.fa.fai, PREFIX.bam, PREFIX.bam.bai and prints a JSON summary (exact algorithmic bytes,
// read-bases, reads) on stdout.
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <map>
#include <string>
#include <thread>
#include <vector>

struct Rng {  // splitmix64 / xoshiro256**
    uint64_t s[4];
    static uint64_t sm(uint64_t& x) { uint64_t z = (x += 0x9e3779b97f4a7c15ull); z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull; z = (z ^ (z >> 27)) * 0x94d049bb133111ebull; return z ^ (z >> 31); }
    explicit Rng(uint64_t seed) { for (auto& v : s) v = sm(seed); }
    static uint64_t rotl(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
    uint64_t next() { uint64_t r = rotl(s[1] * 5, 7) * 9, t = s[1] << 17; s[2] ^= s[0]; s[3] ^= s[1]; s[1] ^= s[2]; s[0] ^= s[3]; s[2] ^= t; s[3] = rotl(s[3], 45); return r; }
    double uni() { return (next() >> 11) * (1.0 / 9007199254740992.0); }
    uint32_t below(uint32_t n) { return (uint32_t)((next() >> 32) * (uint64_t)n >> 32); }
    double normal() { double u = uni(), v = uni(); if (u < 1e-300) u = 1e-300; return std::sqrt(-2 * std::log(u)) * std::cos(6.283185307179586 * v); }
};

struct Contig { std::string name; uint32_t len; std::string seq; std::vector<uint8_t> meth; };

static const char* NT = "ACGT";
static inline char comp(char c) { switch (c) { case 'A': return 'T'; case 'C': return 'G'; case 'G': return 'C'; case 'T': return 'A'; } return 'N'; }

struct Opts {
    std::string out = "synth";
    std::vector<std::pair<std::string, uint32_t>> contigs;
    double coverage = 30;
    uint64_t seed = 20260924ull;
    std::string mods = "m";
    double mean_len = 12000, sigma = 0.6;
    int level = 1, threads = 8;
    bool combined_hm = false, implicit = false, odd = false;
    bool ptags = false;    // --partition-tags: RG:Z (A/B/C or absent), HP (C or i, or absent), XF:f on some reads
    bool long_rg = false;  // --long-rg: the RG values are long run ids (ONT style, ~80 characters) ending in A/B/C
    int64_t win_start = -1, win_end = -1;
    bool duplex = false;       // --duplex: opposite-strand CpG lists (G-h?, G-m?) beside the C+ lists
    uint32_t start_grid = 0;   // --start-grid G: read starts snapped down to multiples of G (amplicon-like stacks of reads with one start)
};

// ---- BGZF / BAM / BAI writing ----------------------------------------------------------------------
static void bgzf_member(const uint8_t* src, size_t n, int level, std::vector<uint8_t>* out) {
    size_t base = out->size();
    out->resize(base + 18 + compressBound(n) + 64 + 8);
    uint8_t* p = out->data() + base;
    const uint8_t hdr[16] = {31, 139, 8, 4, 0, 0, 0, 0, 0, 255, 6, 0, 66, 67, 2, 0};
    memcpy(p, hdr, 16);
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    deflateInit2(&zs, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY);
    zs.next_in = (Bytef*)src; zs.avail_in = (uInt)n;
    zs.next_out = p + 18; zs.avail_out = (uInt)(out->size() - base - 18 - 8);
    deflate(&zs, Z_FINISH);
    size_t clen = zs.total_out;
    deflateEnd(&zs);
    uint16_t bsize = (uint16_t)(clen + 25);
    memcpy(p + 16, &bsize, 2);
    uint32_t crc = (uint32_t)crc32(crc32(0, nullptr, 0), src, (uInt)n), isz = (uint32_t)n;
    memcpy(p + 18 + clen, &crc, 4);
    memcpy(p + 18 + clen + 4, &isz, 4);
    out->resize(base + 18 + clen + 8);
}

static int reg2bin(int64_t beg, int64_t end) {
    --end;
    if (beg >> 14 == end >> 14) return (int)(((1 << 15) - 1) / 7 + (beg >> 14));
    if (beg >> 17 == end >> 17) return (int)(((1 << 12) - 1) / 7 + (beg >> 17));
    if (beg >> 20 == end >> 20) return (int)(((1 << 9) - 1) / 7 + (beg >> 20));
    if (beg >> 23 == end >> 23) return (int)(((1 << 6) - 1) / 7 + (beg >> 23));
    if (beg >> 26 == end >> 26) return (int)(((1 << 3) - 1) / 7 + (beg >> 26));
    return 0;
}

struct RecMeta { int32_t tid, pos, end; uint16_t flag; uint32_t size; };   // size includes the 4-byte block_size

struct TileOut { std::vector<uint8_t> bytes; std::vector<RecMeta> recs; uint64_t alg_bytes = 0, read_bases = 0; };

template <class T> static void put(std::vector<uint8_t>& v, T x) { size_t o = v.size(); v.resize(o + sizeof(T)); memcpy(v.data() + o, &x, sizeof(T)); }

// one read starting at ref position `start` on contig c
static void make_read(const Opts& o, const Contig& c, int32_t tid, uint32_t start, uint64_t read_id, Rng& rng, TileOut* out) {
    double ln = std::log(o.mean_len) + o.sigma * rng.normal();
    uint32_t want = (uint32_t)std::min(200000.0, std::max(500.0, std::exp(ln)));
    const bool rev = rng.uni() < 0.5;
    std::string seq;          // as stored in BAM (reference orientation)
    std::vector<uint32_t> cigar;
    std::vector<int64_t> q2r; // per stored base: reference position or -1
    auto push_op = [&](uint32_t op, uint32_t len) { if (!len) return; if (!cigar.empty() && (cigar.back() & 15) == op) cigar.back() += len << 4; else cigar.push_back(len << 4 | op); };
    const bool clip_l = rng.uni() < 0.15, clip_r = rng.uni() < 0.15;
    if (clip_l) { for (int i = 0; i < 20; i++) { seq.push_back(NT[rng.below(4)]); q2r.push_back(-1); } push_op(4, 20); }
    uint32_t r = start, made = 0;
    bool first = true;
    while (made < want && r < c.len) {
        double u = rng.uni();
        if (!first && u < 0.005) { uint32_t n = 1 + rng.below(3); for (uint32_t i = 0; i < n; i++) { seq.push_back(NT[rng.below(4)]); q2r.push_back(-1); } push_op(1, n); made += n; }
        else if (!first && u < 0.010) { uint32_t n = 1 + rng.below(3); n = std::min(n, c.len - r); if (r + n >= c.len) break; push_op(2, n); r += n; }
        else {
            char b = c.seq[r];
            if (u > 0.99) { char nb; do { nb = NT[rng.below(4)]; } while (nb == b); b = nb; }
            seq.push_back(b); q2r.push_back(r); push_op(0, 1); r++; made++;
        }
        first = false;
    }
    // a read must end on a match for a valid alignment
    while (!cigar.empty() && ((cigar.back() & 15) == 1 || (cigar.back() & 15) == 2)) {
        uint32_t op = cigar.back() & 15, len = cigar.back() >> 4;
        if (op == 1) { seq.resize(seq.size() - len); q2r.resize(q2r.size() - len); } else r -= len;
        cigar.pop_back();
    }
    if (seq.empty() || cigar.empty()) return;
    const uint32_t ref_end = r;
    if (clip_r) { for (int i = 0; i < 20; i++) { seq.push_back(NT[rng.below(4)]); q2r.push_back(-1); } push_op(4, 20); }
    const uint32_t L = (uint32_t)seq.size();
    // a read outside the --region-only window is generated all the same (it consumes its share of the tile's random stream, so
    // the reads of the window are the same reads as in the full file) and only not written
    const bool emit_read = !(o.win_start >= 0 && !((int64_t)start < o.win_end && (int64_t)ref_end > o.win_start));

    // forward (as sequenced) view
    auto fwd = [&](uint32_t f) -> char { return rev ? comp(seq[L - 1 - f]) : seq[f]; };
    auto fwd_ref = [&](uint32_t f) -> int64_t { return rev ? q2r[L - 1 - f] : q2r[f]; };
    // MM / ML
    std::string mm;
    std::vector<uint8_t> ml;
    uint16_t flag = rev ? 16 : 0;
    bool with_tags = true;
    bool mn_tag = false;
    if (o.odd) {
        double u = rng.uni();
        if (u < 0.01) flag |= 0x100; else if (u < 0.02) flag |= 0x800; else if (u < 0.03) flag |= 0x400; else if (u < 0.04) flag |= 0x200;
        else if (u < 0.06) with_tags = false;
        else if (u < 0.10) mn_tag = true;
    }
    const char mode = o.implicit ? '.' : '?';
    if (with_tags) {
        const bool want_h = o.mods.find('h') != std::string::npos, want_m = o.mods.find('m') != std::string::npos, want_a = o.mods.find('a') != std::string::npos;
        if (want_h || want_m) {
            // CpG calls in read orientation
            std::vector<uint32_t> deltas;
            std::vector<uint8_t> qh, qm;
            uint32_t skipped = 0;
            for (uint32_t f = 0; f < L; f++) {
                if (fwd(f) != 'C') continue;
                const bool cpg = f + 1 < L && fwd(f + 1) == 'G';
                if (!cpg) { skipped++; continue; }
                deltas.push_back(skipped);
                skipped = 0;
                int64_t rp = fwd_ref(f);
                double level = 0.5;
                if (rp >= 0) { uint32_t cpos = rev ? (uint32_t)rp - 1 : (uint32_t)rp; if (cpos < c.len) level = c.meth[cpos] / 255.0; }
                const bool confident = rng.uni() < 0.8;
                const bool is_mod = rng.uni() < level;
                const bool is_h = want_h && is_mod && rng.uni() < 0.15;
                uint32_t qa, qb;   // qa: called-state probability byte, qb: the other
                if (confident) { qa = 230 + rng.below(26); qb = rng.below(256 - qa); } else { qa = rng.below(256); qb = rng.below(256 - qa); }
                if (!is_mod) { uint32_t lo = rng.below(26); qa = confident ? lo : qa; qb = confident ? rng.below(26) : qb; if (qa + qb > 255) qb = 255 - qa; }
                if (want_h && want_m) { if (is_h) { qh.push_back((uint8_t)qa); qm.push_back((uint8_t)qb); } else { qm.push_back((uint8_t)qa); qh.push_back((uint8_t)qb); } }
                else if (want_m) qm.push_back((uint8_t)qa);
                else qh.push_back((uint8_t)qa);
            }
            auto emit = [&](const std::string& hdr, const std::vector<uint8_t>* a, const std::vector<uint8_t>* b) {
                mm += hdr;
                char buf[16];
                for (uint32_t d : deltas) { int n = snprintf(buf, sizeof buf, ",%u", d); mm.append(buf, n); }
                mm += ';';
                for (size_t i = 0; i < deltas.size(); i++) { ml.push_back((*a)[i]); if (b) ml.push_back((*b)[i]); }
            };
            if (want_h && want_m) {
                if (o.combined_hm) emit(std::string("C+hm") + mode, &qh, &qm);
                else { emit(std::string("C+h") + mode, &qh, nullptr); emit(std::string("C+m") + mode, &qm, nullptr); }
            } else if (want_m) emit(std::string("C+m") + mode, &qm, nullptr);
            else emit(std::string("C+h") + mode, &qh, nullptr);
            if (o.duplex) {
                // the G of every CpG in read orientation: a call on the C of the opposite strand, drawn independently of the C+ call
                std::vector<uint8_t> gh, gm;
                deltas.clear();
                skipped = 0;
                for (uint32_t f = 0; f < L; f++) {
                    if (fwd(f) != 'G') continue;
                    if (!(f > 0 && fwd(f - 1) == 'C')) { skipped++; continue; }
                    deltas.push_back(skipped);
                    skipped = 0;
                    const int64_t rp = fwd_ref(f);
                    double level = 0.5;
                    if (rp >= 0) { const uint32_t cpos = rev ? (uint32_t)rp : (uint32_t)rp - 1; if (cpos < c.len) level = c.meth[cpos] / 255.0; }
                    const bool is_mod = rng.uni() < level;
                    const bool is_h = want_h && is_mod && rng.uni() < 0.2;
                    uint32_t qa = 225 + rng.below(31), qb = rng.below(256 - qa);
                    if (!is_mod) { qa = rng.below(30); qb = rng.below(30); }
                    if (want_h && want_m) { if (is_h) { gh.push_back((uint8_t)qa); gm.push_back((uint8_t)qb); } else { gm.push_back((uint8_t)qa); gh.push_back((uint8_t)qb); } }
                    else if (want_m) gm.push_back((uint8_t)qa);
                    else gh.push_back((uint8_t)qa);
                }
                if (want_h) emit(std::string("G-h") + mode, &gh, nullptr);
                if (want_m) emit(std::string("G-m") + mode, &gm, nullptr);
            }
        }
        if (want_a) {
            mm += std::string("A+a") + mode;
            char buf[16];
            uint32_t skipped = 0;
            for (uint32_t f = 0; f < L; f++) {
                if (fwd(f) != 'A') continue;
                if (rng.uni() < 0.02) { skipped++; continue; }   // a few uncalled A's
                int n = snprintf(buf, sizeof buf, ",%u", skipped);
                mm.append(buf, n);
                skipped = 0;
                ml.push_back(rng.uni() < 0.03 ? (uint8_t)(200 + rng.below(56)) : (uint8_t)rng.below(40));
            }
            mm += ';';
        }
    }
    if (!emit_read) return;
    // ---- BAM record
    char name[32];
    int l_name = snprintf(name, sizeof name, "r%010llu", (unsigned long long)read_id) + 1;
    std::vector<uint8_t>& v = out->bytes;
    const size_t rec0 = v.size();
    put<uint32_t>(v, 0);   // block_size placeholder
    put<int32_t>(v, tid); put<int32_t>(v, (int32_t)start);
    v.push_back((uint8_t)l_name); v.push_back(60);
    put<uint16_t>(v, (uint16_t)reg2bin(start, ref_end));
    put<uint16_t>(v, (uint16_t)cigar.size()); put<uint16_t>(v, flag); put<int32_t>(v, (int32_t)L);
    put<int32_t>(v, -1); put<int32_t>(v, -1); put<int32_t>(v, 0);
    v.insert(v.end(), name, name + l_name);
    for (uint32_t c4 : cigar) put<uint32_t>(v, c4);
    auto nib = [](char b) -> uint8_t { switch (b) { case 'A': return 1; case 'C': return 2; case 'G': return 4; case 'T': return 8; } return 15; };
    for (uint32_t i = 0; i < L; i += 2) v.push_back((uint8_t)(nib(seq[i]) << 4 | (i + 1 < L ? nib(seq[i + 1]) : 0)));
    v.insert(v.end(), L, 0xff);
    if (with_tags) {
        if (mn_tag) { v.push_back('M'); v.push_back('N'); v.push_back('i'); put<int32_t>(v, (int32_t)L); }
        v.push_back('M'); v.push_back('M'); v.push_back('Z'); v.insert(v.end(), mm.begin(), mm.end()); v.push_back(0);
        v.push_back('M'); v.push_back('L'); v.push_back('B'); v.push_back('C'); put<uint32_t>(v, (uint32_t)ml.size()); v.insert(v.end(), ml.begin(), ml.end());
    }
    if (o.ptags) {
        const double u1 = rng.uni(), u2 = rng.uni(), u3 = rng.uni();
        if (u1 < 0.9) {
            v.push_back('R'); v.push_back('G'); v.push_back('Z');
            if (o.long_rg) { const char* run = "4524e8b9-b90e-4ffb-a13a-380266513b64_dna_r10.4.1_e8.2_400bps_hac@v4.2.0_barcode0"; v.insert(v.end(), run, run + strlen(run)); }
            v.push_back((uint8_t)("ABC"[(int)(u1 * 10) % 3])); v.push_back(0);
        }
        if (u2 < 0.7) { v.push_back('H'); v.push_back('P'); v.push_back('C'); v.push_back((uint8_t)(u2 < 0.35 ? 1 : 2)); }
        else if (u2 < 0.8) { v.push_back('H'); v.push_back('P'); v.push_back('i'); put<int32_t>(v, 3); }
        if (u3 < 0.3) { v.push_back('X'); v.push_back('F'); v.push_back('f'); const float f = u3 < 0.1 ? 0.1f : (u3 < 0.2 ? 2.5f : 1.0f / 3.0f); uint32_t b; memcpy(&b, &f, 4); put<uint32_t>(v, b); }
    }
    const uint32_t bs = (uint32_t)(v.size() - rec0 - 4);
    memcpy(v.data() + rec0, &bs, 4);
    out->recs.push_back({tid, (int32_t)start, (int32_t)ref_end, flag, bs + 4});
    out->alg_bytes += 32 + 4ull * cigar.size() + (L + 1) / 2 + (with_tags ? mm.size() + ml.size() : 0);
    out->read_bases += L;
}

int main(int argc, char** argv) {
    Opts o;
    for (int i = 1; i < argc; i++) {
        std::string a = argv[i];
        auto val = [&]() { if (i + 1 >= argc) { fprintf(stderr, "missing value for %s\n", a.c_str()); exit(2); } return std::string(argv[++i]); };
        if (a == "--out") o.out = val();
        else if (a == "--contig") { std::string s = val(); auto c = s.find(':'); o.contigs.push_back({s.substr(0, c), (uint32_t)std::stoul(s.substr(c + 1))}); }
        else if (a == "--coverage") o.coverage = std::stod(val());
        else if (a == "--seed") o.seed = std::stoull(val());
        else if (a == "--mods") o.mods = val();
        else if (a == "--mean-len") o.mean_len = std::stod(val());
        else if (a == "--level") o.level = std::stoi(val());
        else if (a == "--threads") o.threads = std::stoi(val());
        else if (a == "--combined-hm") o.combined_hm = true;
        else if (a == "--implicit") o.implicit = true;
        else if (a == "--odd-records") o.odd = true;
        else if (a == "--partition-tags") o.ptags = true;
        else if (a == "--long-rg") o.long_rg = true;
        else if (a == "--duplex") o.duplex = true;
        else if (a == "--start-grid") o.start_grid = (uint32_t)std::stoul(val());
        else if (a == "--region-only") { std::string s = val(); auto d = s.find('-'); o.win_start = std::stoll(s.substr(0, d)); o.win_end = std::stoll(s.substr(d + 1)); }
        else { fprintf(stderr, "unknown flag %s\n", a.c_str()); return 2; }
    }
    if (o.contigs.empty()) o.contigs.push_back({"syn1", 1000000});
    const int nt = std::max(1, o.threads);

    // ---- reference: uniform ACGT, CpG observed/expected 0.25, per-site methylation ~ Beta(0.5,0.5)
    std::vector<Contig> contigs(o.contigs.size());
    for (size_t ci = 0; ci < contigs.size(); ci++) {
        Contig& c = contigs[ci];
        c.name = o.contigs[ci].first; c.len = o.contigs[ci].second;
        c.seq.resize(c.len); c.meth.assign(c.len, 0);
        const uint32_t TILE = 1u << 20;
        const uint32_t ntile = (c.len + TILE - 1) / TILE;
        std::atomic<uint32_t> next{0};
        auto work = [&]() {
            for (;;) {
                uint32_t t = next.fetch_add(1);
                if (t >= ntile) break;
                Rng rng(o.seed * 0x9e3779b97f4a7c15ull + ci * 1000003ull + t);
                uint32_t b = t * TILE, e = std::min(c.len, b + TILE);
                char prev = 'A';
                for (uint32_t i = b; i < e; i++) {
                    char ch = NT[rng.below(4)];
                    if (prev == 'C' && ch == 'G' && rng.uni() >= 0.25) { do { ch = NT[rng.below(4)]; } while (ch == 'G'); }
                    c.seq[i] = ch;
                    prev = ch;
                }
            }
        };
        std::vector<std::thread> th;
        for (int t = 1; t < nt; t++) th.emplace_back(work);
        work();
        for (auto& t : th) t.join();
        Rng mr(o.seed ^ (0xabcdefull + ci));
        for (uint32_t i = 0; i + 1 < c.len; i++) if (c.seq[i] == 'C' && c.seq[i + 1] == 'G') {
            double u = mr.uni(); double s = std::sin(1.5707963267948966 * u); c.meth[i] = (uint8_t)(255.0 * s * s);   // arcsine law == Beta(.5,.5)
        }
    }
    {   // FASTA + fai
        FILE* f = fopen((o.out + ".fa").c_str(), "wb");
        FILE* fi = fopen((o.out + ".fa.fai").c_str(), "wb");
        if (!f || !fi) { fprintf(stderr, "cannot write %s.fa\n", o.out.c_str()); return 1; }
        uint64_t off = 0;
        for (auto& c : contigs) {
            off += fprintf(f, ">%s\n", c.name.c_str());
            fprintf(fi, "%s\t%u\t%llu\t60\t61\n", c.name.c_str(), c.len, (unsigned long long)off);
            for (uint32_t i = 0; i < c.len; i += 60) { uint32_t n = std::min(60u, c.len - i); fwrite(c.seq.data() + i, 1, n, f); fputc('\n', f); off += n + 1; }
        }
        fclose(f); fclose(fi);
    }
    // ---- reads per 256 kb start tile (independent streams => deterministic regardless of thread count)
    struct TileId { uint32_t ci, t; };
    std::vector<TileId> tiles;
    const uint32_t RT = 1u << 18;
    for (uint32_t ci = 0; ci < contigs.size(); ci++) for (uint32_t t = 0; t < (contigs[ci].len + RT - 1) / RT; t++) tiles.push_back({ci, t});
    std::vector<TileOut> outs(tiles.size());
    // mean stored length of the clipped lognormal is a little above mean_len*exp(sigma^2/2); starts per base = coverage / E[len]
    const double e_len = o.mean_len * std::exp(o.sigma * o.sigma / 2);
    {
        std::atomic<size_t> next{0};
        auto work = [&]() {
            for (;;) {
                size_t k = next.fetch_add(1);
                if (k >= tiles.size()) break;
                const Contig& c = contigs[tiles[k].ci];
                uint32_t b = tiles[k].t * RT, e = std::min(c.len, b + RT);
                if (o.win_start >= 0 && ((int64_t)b >= o.win_end || (int64_t)e + 250000 < o.win_start)) continue;
                Rng rng((o.seed + 77) * 0xd1342543de82ef95ull + tiles[k].ci * 7919ull + tiles[k].t);
                double expect = o.coverage * (e - b) / e_len;
                uint32_t n = (uint32_t)expect + (rng.uni() < expect - std::floor(expect) ? 1 : 0);
                std::vector<uint32_t> starts(n);
                for (auto& s : starts) { s = b + rng.below(e - b); if (o.start_grid) s = std::max(b, s / o.start_grid * o.start_grid); }
                std::sort(starts.begin(), starts.end());
                uint64_t rid = ((uint64_t)tiles[k].ci << 40) | ((uint64_t)tiles[k].t << 20);
                for (uint32_t s : starts) make_read(o, c, (int32_t)tiles[k].ci, s, rid++, rng, &outs[k]);
            }
        };
        std::vector<std::thread> th;
        for (int t = 1; t < nt; t++) th.emplace_back(work);
        work();
        for (auto& t : th) t.join();
    }
    // ---- serialise: header, then records; BGZF members of <= 0xff00 bytes (records may span members)
    std::vector<uint8_t> head;
    std::string text = "@HD\tVN:1.6\tSO:coordinate\n";
    for (auto& c : contigs) text += "@SQ\tSN:" + c.name + "\tLN:" + std::to_string(c.len) + "\n";
    head.insert(head.end(), {'B', 'A', 'M', 1});
    put<uint32_t>(head, (uint32_t)text.size()); head.insert(head.end(), text.begin(), text.end());
    put<uint32_t>(head, (uint32_t)contigs.size());
    for (auto& c : contigs) { put<uint32_t>(head, (uint32_t)c.name.size() + 1); head.insert(head.end(), c.name.begin(), c.name.end()); head.push_back(0); put<uint32_t>(head, c.len); }
    // uncompressed offsets of every tile
    std::vector<uint64_t> tile_off(outs.size() + 1);
    uint64_t total = head.size();
    for (size_t k = 0; k < outs.size(); k++) { tile_off[k] = total; total += outs[k].bytes.size(); }
    tile_off[outs.size()] = total;
    const uint64_t MEMBER = 0xff00;
    const uint64_t n_member = (total + MEMBER - 1) / MEMBER;
    auto copy_range = [&](uint64_t b, uint64_t e, uint8_t* dst) {   // gather [b,e) of the virtual stream
        uint64_t at = b;
        if (at < head.size()) { uint64_t n = std::min<uint64_t>(e, head.size()) - at; memcpy(dst, head.data() + at, n); dst += n; at += n; }
        if (at >= e) return;
        size_t k = std::upper_bound(tile_off.begin(), tile_off.end(), at) - tile_off.begin() - 1;
        while (at < e) {
            while (k + 1 < tile_off.size() && tile_off[k + 1] <= at) k++;
            uint64_t n = std::min(e, tile_off[k + 1]) - at;
            memcpy(dst, outs[k].bytes.data() + (at - tile_off[k]), n);
            dst += n; at += n;
        }
    };
    // compress members in parallel, groups of 256 members per task
    const uint64_t GROUP = 256;
    const uint64_t n_group = (n_member + GROUP - 1) / GROUP;
    std::vector<std::vector<uint8_t>> gbytes(n_group);
    std::vector<std::vector<uint32_t>> gsizes(n_group);
    {
        std::atomic<uint64_t> next{0};
        auto work = [&]() {
            std::vector<uint8_t> buf(MEMBER);
            for (;;) {
                uint64_t g = next.fetch_add(1);
                if (g >= n_group) break;
                for (uint64_t m = g * GROUP; m < std::min(n_member, (g + 1) * GROUP); m++) {
                    uint64_t b = m * MEMBER, e = std::min(total, b + MEMBER);
                    copy_range(b, e, buf.data());
                    size_t before = gbytes[g].size();
                    bgzf_member(buf.data(), e - b, o.level, &gbytes[g]);
                    gsizes[g].push_back((uint32_t)(gbytes[g].size() - before));
                }
            }
        };
        std::vector<std::thread> th;
        for (int t = 1; t < nt; t++) th.emplace_back(work);
        work();
        for (auto& t : th) t.join();
    }
    std::vector<uint64_t> member_coff(n_member + 1, 0);
    {
        FILE* f = fopen((o.out + ".bam").c_str(), "wb");
        if (!f) { fprintf(stderr, "cannot write %s.bam\n", o.out.c_str()); return 1; }
        uint64_t coff = 0, m = 0;
        for (uint64_t g = 0; g < n_group; g++) {
            fwrite(gbytes[g].data(), 1, gbytes[g].size(), f);
            for (uint32_t sz : gsizes[g]) { member_coff[m++] = coff; coff += sz; }
        }
        member_coff[n_member] = coff;
        static const uint8_t eof[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 0x42, 0x43, 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
        fwrite(eof, 1, 28, f);
        fclose(f);
    }
    auto voff = [&](uint64_t u) -> uint64_t { uint64_t m = u / MEMBER; if (m >= n_member) return member_coff[n_member] << 16; return member_coff[m] << 16 | (u % MEMBER); };
    // ---- BAI
    {
        struct RefIdx { std::map<uint32_t, std::vector<std::pair<uint64_t, uint64_t>>> bins; std::vector<uint64_t> lin; uint64_t beg = ~0ull, end = 0, n_map = 0, n_unmap = 0; };
        std::vector<RefIdx> idx(contigs.size());
        for (size_t k = 0; k < outs.size(); k++) {
            uint64_t u = tile_off[k];
            for (auto& r : outs[k].recs) {
                RefIdx& R = idx[r.tid];
                uint64_t vb = voff(u), ve = voff(u + r.size);
                uint32_t bin = (uint32_t)reg2bin(r.pos, r.end);
                auto& ch = R.bins[bin];
                if (!ch.empty() && ch.back().second >> 16 == vb >> 16) ch.back().second = ve; else ch.push_back({vb, ve});
                for (uint32_t w = (uint32_t)r.pos >> 14; w <= (uint32_t)(r.end - 1) >> 14; w++) { if (R.lin.size() <= w) R.lin.resize(w + 1, 0); if (!R.lin[w]) R.lin[w] = vb; }
                R.beg = std::min(R.beg, vb); R.end = std::max(R.end, ve);
                if (r.flag & 4) R.n_unmap++; else R.n_map++;
                u += r.size;
            }
        }
        std::vector<uint8_t> b;
        b.insert(b.end(), {'B', 'A', 'I', 1});
        put<uint32_t>(b, (uint32_t)contigs.size());
        for (auto& R : idx) {
            const bool any = R.n_map + R.n_unmap > 0;
            put<uint32_t>(b, (uint32_t)R.bins.size() + (any ? 1 : 0));
            for (auto& kv : R.bins) { put<uint32_t>(b, kv.first); put<uint32_t>(b, (uint32_t)kv.second.size()); for (auto& c : kv.second) { put<uint64_t>(b, c.first); put<uint64_t>(b, c.second); } }
            if (any) { put<uint32_t>(b, 37450u); put<uint32_t>(b, 2u); put<uint64_t>(b, R.beg); put<uint64_t>(b, R.end); put<uint64_t>(b, R.n_map); put<uint64_t>(b, R.n_unmap); }
            for (size_t w = 1; w < R.lin.size(); w++) if (!R.lin[w]) R.lin[w] = R.lin[w - 1];
            put<uint32_t>(b, (uint32_t)R.lin.size());
            for (uint64_t v : R.lin) put<uint64_t>(b, v);
        }
        put<uint64_t>(b, 0ull);
        FILE* f = fopen((o.out + ".bam.bai").c_str(), "wb");
        fwrite(b.data(), 1, b.size(), f);
        fclose(f);
    }
    uint64_t alg = 0, bases = 0, reads = 0, positions = 0;
    for (auto& t : outs) { alg += t.alg_bytes; bases += t.read_bases; reads += t.recs.size(); }
    for (auto& c : contigs) positions += c.len;
    printf("{\"reads\": %llu, \"read_bases\": %llu, \"algorithmic_input_bytes\": %llu, \"positions\": %llu, \"bam_bytes\": %llu}\n",
           (unsigned long long)reads, (unsigned long long)bases, (unsigned long long)alg, (unsigned long long)positions, (unsigned long long)member_coff[n_member] + 28);
    return 0;
}
