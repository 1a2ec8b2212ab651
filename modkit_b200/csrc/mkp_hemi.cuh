// `modkit pileup-hemi` on the device (sm_100a): the pair and row kernels that follow the pileup decode (k_parse, k_resolve).
//
// The chunk is uploaded with two bitmaps: focus_pos = the hemi columns (positive-strand motif positions of the intervals),
// focus_neg = their partner positions (column + motif offset). k_parse / k_resolve run unchanged and leave every read's call
// records (reference position, mod strand, MM base, threshold state) in `calls`; nothing here re-decodes MM/ML.
//   k_hemi_pairs  warp per read (longest-first queue): walks the read's CIGAR over the columns in its span and adds one
//                 feature per column: deletion, or the (top, bottom) call pair of DuplexReadCache::get_duplex_mod_call
//                 (src/read_cache.rs:368-463, src/mod_bam.rs:1674-1830), or NoCall; skip-set reads add one NoCall per
//                 interval at their first column there (src/pileup/duplex.rs:238-339 with the per-interval read cache)
//   k_hemi_rows   thread per column word: DuplexFeatureVector::decode (src/pileup/duplex.rs:84-205), rows in output order
#pragma once
#include "mkp_kernels.cuh"

namespace mkp {

constexpr int HEMI_MAX_PATTERNS = 256;     // registry size; a chunk with more distinct (base, top, bottom) patterns is an error
constexpr int HS_DEL = 0;                  // per-column counter slot: n_delete
constexpr int HS_FAIL = 1;                 // [pb]
constexpr int HS_NOCALL = 5;               // [pb]
constexpr int HS_PAT = 9;                  // [pattern id], `pat_cap` of them
constexpr uint32_t HEMI_ANY_MOD = 33;      // half code of --combine-mods: the any-mod code of the primary base

// pattern key: primary base (2 bits) | top half << 2 | bottom half << 8; a half is 0 (canonical), 1 + state id, or HEMI_ANY_MOD
__device__ __forceinline__ uint32_t hemi_key(uint32_t pb, uint32_t top, uint32_t bot) { return pb | (top << 2) | (bot << 8); }

struct HemiDev {
    const mkp_read_hdr* hdrs;
    const uint8_t* heap;
    const ReadMeta* meta;
    const uint2* calls;
    uint32_t n_reads, cs, ce;
    const uint32_t* cols;           // focus_pos: the hemi columns
    const uint32_t* col_prefix;     // columns before each bitmap word
    int32_t offset;                 // partner = column + offset (MotifInfo::offset, src/find_motifs/motif_bed.rs:111-141)
    const uint32_t* iv_starts;      // interval starts of the chunk, ascending
    uint32_t n_iv;
    uint32_t* slots;                // per column: HS_PAT + pat_cap words
    uint32_t stride, pat_cap;
    uint32_t* pat_keys;             // registry [HEMI_MAX_PATTERNS], ~0 = empty
    uint32_t* n_pat;                // entries used (> HEMI_MAX_PATTERNS: overflow)
    uint32_t* work;                 // dynamic read counter
    const uint32_t* order;          // longest reads first, or null
    uint32_t combine;               // --combine-mods
};

__device__ __noinline__ uint32_t hemi_pattern_id(const HemiDev& H, uint32_t key) {
    for (uint32_t i = 0; i < (uint32_t)HEMI_MAX_PATTERNS; i++) {
        uint32_t k = *((volatile uint32_t*)H.pat_keys + i);
        if (k == 0xffffffffu) {
            k = atomicCAS(H.pat_keys + i, 0xffffffffu, key);
            if (k == 0xffffffffu) { atomicMax(H.n_pat, i + 1); return i; }
        }
        if (k == key) return i;
    }
    atomicMax(H.n_pat, (uint32_t)HEMI_MAX_PATTERNS + 1);
    return 0xffffffffu;
}

__device__ __forceinline__ bool hemi_edge_keep(uint32_t f, uint32_t L) {
    if (!c_par.edge_on) return true;
    return c_par.edge_inv ? (f < c_par.edge_start || f >= L - c_par.edge_end) : (f >= c_par.edge_start && f < L - c_par.edge_end);
}

// query position aligned to reference position r (M/=/X), or ~0: a serial walk over the read's CIGAR (partners outside the batch
// of ops in shared memory whose implicit table has to be consulted - rare)
__device__ __noinline__ uint32_t hemi_query_at(const uint32_t* cig, uint32_t n_cigar, uint32_t ref_start, uint32_t r) {
    uint32_t qc = 0, rc = ref_start;
    for (uint32_t i = 0; i < n_cigar; i++) {
        const uint32_t c = cig[i], op = c & 15, len = c >> 4;
        const bool rl = op == 0 || op == 2 || op == 3 || op == 7 || op == 8;
        if (rl && r < rc + len) return (op == 0 || op == 7 || op == 8) ? qc + (r - rc) : 0xffffffffu;
        if (op == 0 || op == 1 || op == 4 || op == 7 || op == 8) qc += len;
        if (rl) rc += len;
        if (rc > r) break;
    }
    return 0xffffffffu;
}

__global__ void __launch_bounds__(256) k_hemi_pairs(HemiDev H) {
    __shared__ uint32_t s_op[8][32], s_q[8][32], s_r[8][33];
    const uint32_t lane = lane_id();
    const uint32_t wib = threadIdx.x >> 5;
    for (;;) {
        uint32_t ri = 0;
        if (lane == 0) { ri = atomicAdd(H.work, 1u); if (H.order && ri < H.n_reads) ri = H.order[ri]; }
        ri = __shfl_sync(FULL, ri, 0);
        if (ri >= H.n_reads) break;
        const ReadMeta m = H.meta[ri];
        if (!(m.flags & 1)) continue;                                  // not admitted by the pileup (flags, seq_len == 0)
        const mkp_read_hdr h = H.hdrs[ri];
        if ((uint32_t)m.ref_end <= H.cs || (uint32_t)h.ref_start >= H.ce) continue;
        const uint32_t a = (h.flags & 0x10) ? 1u : 0u;
        const uint32_t L = h.l_seq;
        const uint32_t* cig = (const uint32_t*)(H.heap + h.off);
        const uint8_t* seq = H.heap + h.off + 4ull * h.n_cigar;
        const bool has_mods = m.flags & 2;                            // else: the skip set
        const uint2* rcalls = H.calls + m.entry_off;
        const uint32_t n_calls = has_mods ? m.n_calls : 0u;
        uint32_t last_iv = 0xffffffffu;                               // skip set: interval of the last NoCall
        uint32_t qc = 0, rc = (uint32_t)h.ref_start;
        for (uint32_t b0 = 0; b0 < h.n_cigar; b0 += 32) {
            const uint32_t i = b0 + lane;
            const uint32_t c = i < h.n_cigar ? cig[i] : 0;
            const uint32_t op = c & 15, len = c >> 4;
            const uint32_t ql = (op == 0 || op == 1 || op == 4 || op == 7 || op == 8) ? len : 0;
            const uint32_t rl = (op == 0 || op == 2 || op == 3 || op == 7 || op == 8) ? len : 0;
            const uint32_t qi = warp_incl_scan(ql), rr = warp_incl_scan(rl);
            const uint32_t q0 = qc + qi - ql, r0 = rc + rr - rl;
            qc += __shfl_sync(FULL, qi, 31);
            rc += __shfl_sync(FULL, rr, 31);
            const uint32_t R0 = __shfl_sync(FULL, r0, 0), R1 = rc;
            __syncwarp();
            s_op[wib][lane] = op | (len << 4); s_q[wib][lane] = q0; s_r[wib][lane] = r0;
            if (lane == 0) s_r[wib][32] = R1;
            __syncwarp();
            const uint32_t blo = R0 > H.cs ? R0 : H.cs, bhi = R1 < H.ce ? R1 : H.ce;
            if (blo >= bhi) continue;
            const uint32_t w_first = (blo - H.cs) >> 5, w_last = (bhi - 1 - H.cs) >> 5;
            for (uint32_t wt = w_first; wt <= w_last; wt += 32) {
                // lane per bitmap word, then the columns of these 32 words in rounds of 32 (lane per column, ascending)
                const uint32_t w = wt + lane;
                uint32_t bits = 0;
                if (w <= w_last) {
                    bits = H.cols[w];
                    const uint32_t wbase = H.cs + (w << 5);
                    if (blo > wbase) bits &= FULL << (blo - wbase);
                    if (bhi < wbase + 32) bits &= (1u << (bhi - wbase)) - 1u;
                }
                const uint32_t cnt = __popc(bits), incl = warp_incl_scan(cnt), total = __shfl_sync(FULL, incl, 31);
                for (uint32_t c0 = 0; c0 < total; c0 += 32) {
                    const uint32_t ci = c0 + lane;
                    const bool act = ci < total;
                    // word lane holding column ci: first lane whose inclusive count exceeds ci
                    uint32_t k = 0;
#pragma unroll
                    for (int stp = 16; stp >= 1; stp >>= 1) { const uint32_t v = __shfl_sync(FULL, incl, k + stp - 1); if (v <= ci) k += stp; }
                    const uint32_t wb = __shfl_sync(FULL, bits, k & 31), ex = __shfl_sync(FULL, incl - cnt, k & 31);
                    uint32_t p = 0, kind = 0, q = 0;                   // kind: 0 none, 1 deletion, 2 base
                    uint32_t slot = 0;
                    if (act) {
                        const uint32_t bit = __fns(wb, 0, (int)(ci - ex) + 1);
                        const uint32_t ww = wt + k;
                        p = H.cs + (ww << 5) + bit;
                        slot = H.col_prefix[ww] + __popc(H.cols[ww] & ((1u << bit) - 1u));
                        uint32_t j = 0;
#pragma unroll
                        for (int stp = 16; stp >= 1; stp >>= 1) if (s_r[wib][j + stp] <= p) j += stp;
                        while (j < 31 && s_r[wib][j + 1] <= p) j++;
                        const uint32_t jc = s_op[wib][j], jop = jc & 15;
                        if (jop == 2) kind = 1;
                        else if (jop == 0 || jop == 7 || jop == 8) { q = s_q[wib][j] + (p - s_r[wib][j]); kind = q < L ? 2u : 0u; }
                    }
                    uint32_t* S = H.slots + (size_t)slot * H.stride;
                    if (kind == 1) atomicAdd(&S[HS_DEL], 1u);          // counted before any read-cache lookup
                    int nb = 4;
                    if (kind == 2) nb = nib_to_base(seq_nibble(seq, q));
                    const bool based = kind == 2 && nb <= 3;          // the stored base is A, C, G or T (get_forward_read_base)
                    const uint32_t pb = based ? (uint32_t)nb : 0u;
                    if (!has_mods) {
                        // skip set: the first column of each interval where the read has a base gets one NoCall
                        uint32_t iv = 0;
                        if (based) {
                            uint32_t lo = 0, hi = H.n_iv;
                            while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (H.iv_starts[mid] <= p) lo = mid; else hi = mid; }
                            iv = lo;
                        }
                        const uint32_t bm = __ballot_sync(FULL, based);
                        const uint32_t below = bm & ((1u << lane) - 1u);
                        const uint32_t src = below ? 31u - __clz(below) : lane;
                        const uint32_t prev_iv = __shfl_sync(FULL, iv, src);
                        if (based && (below ? prev_iv : last_iv) != iv) atomicAdd(&S[HS_NOCALL + pb], 1u);
                        if (bm) last_iv = __shfl_sync(FULL, iv, 31 - __clz(bm));
                        continue;
                    }
                    // the two halves: top = (mod strand a, MM base fb) at p, bottom = (1 - a, comp(fb)) at p + offset
                    const uint32_t fb = a ? 3u - pb : pb;
                    const int64_t pp = (int64_t)p + H.offset;
                    const uint32_t partner = pp >= 0 ? (uint32_t)pp : 0xffffffffu;
                    const uint32_t want_top = a | (fb << 1), want_bot = (1u - a) | ((3u - fb) << 1);
                    uint32_t top = 0xffffffffu, bot = 0xffffffffu;      // state (0 filtered, 1 canonical, 2 + id) or ~0 = none
                    bool need = based;
                    for (uint32_t k0 = 0; k0 < n_calls && __any_sync(FULL, need); k0 += 32) {
                        uint2 rec = make_uint2(0xffffffffu, 0u);
                        if (k0 + lane < n_calls) rec = rcalls[k0 + lane];
                        const uint32_t nt = n_calls - k0 < 32 ? n_calls - k0 : 32;
                        for (uint32_t t = 0; t < nt; t++) {
                            const uint32_t rx = __shfl_sync(FULL, rec.x, t), ry = __shfl_sync(FULL, rec.y, t);
                            if (!need) continue;
                            if (rx == p && (ry & 7u) == want_top) top = (ry >> 3) & 0xffu;
                            if (rx == partner && (ry & 7u) == want_bot) bot = (ry >> 3) & 0xffu;
                        }
                        if (top != 0xffffffffu && (bot != 0xffffffffu || partner == 0xffffffffu)) need = false;
                    }
                    if (!based) continue;
                    // implicit tables: every other occurrence of the table's base is an inferred entry (subject to the edge filter)
                    if (top == 0xffffffffu) {
                        const uint32_t imp = (m.imp[a] >> (8 * fb)) & 0xffu;
                        if ((imp & 0x80u) && hemi_edge_keep(a ? L - 1u - q : q, L)) top = imp & 0x7fu;
                    }
                    if (bot == 0xffffffffu && partner != 0xffffffffu) {
                        const uint32_t imp = (m.imp[1 - a] >> (8 * (3u - fb))) & 0xffu;
                        if ((imp & 0x80u) && partner >= (uint32_t)h.ref_start && partner < (uint32_t)m.ref_end) {
                            uint32_t q2 = 0xffffffffu;
                            if (partner >= R0 && partner < R1) {
                                uint32_t j = 0;
                                while (j < 31 && s_r[wib][j + 1] <= partner) j++;
                                const uint32_t jop = s_op[wib][j] & 15;
                                if (jop == 0 || jop == 7 || jop == 8) q2 = s_q[wib][j] + (partner - s_r[wib][j]);
                            } else q2 = hemi_query_at(cig, h.n_cigar, (uint32_t)h.ref_start, partner);
                            if (q2 < L) {
                                const int nb2 = nib_to_base(seq_nibble(seq, q2));
                                const uint32_t fb2 = nb2 > 3 ? 4u : (a ? 3u - (uint32_t)nb2 : (uint32_t)nb2);
                                if (fb2 == 3u - fb && hemi_edge_keep(a ? L - 1u - q2 : q2, L)) bot = imp & 0x7fu;
                            }
                        }
                    }
                    if (top == 0xffffffffu || bot == 0xffffffffu) { atomicAdd(&S[HS_NOCALL + pb], 1u); continue; }
                    if (top == 0 || bot == 0) { atomicAdd(&S[HS_FAIL + pb], 1u); continue; }
                    const uint32_t th = top == 1 ? 0u : (H.combine ? HEMI_ANY_MOD : top - 1u);
                    const uint32_t bh = bot == 1 ? 0u : (H.combine ? HEMI_ANY_MOD : bot - 1u);
                    const uint32_t id = hemi_pattern_id(H, hemi_key(pb, th, bh));
                    if (id < H.pat_cap) atomicAdd(&S[HS_PAT + id], 1u);
                }
            }
            __syncwarp();
        }
    }
}

struct HemiRowDev {
    const uint32_t* cols; const uint32_t* col_prefix;
    uint32_t n_words, cs;
    const uint32_t* slots;
    uint32_t stride, n_pat;
    const uint32_t* pat_keys;
    const unsigned long long* states;
    uint32_t* row_counts;     // per bitmap word
    const uint32_t* row_prefix;
    mkp_hemi_row* rows;
};

__device__ __forceinline__ uint32_t hemi_half_code(const HemiRowDev& R, uint32_t pb, uint32_t h) {
    return h == 0 ? 0u : h == HEMI_ANY_MOD ? (uint32_t)("ACGT"[pb]) : (uint32_t)R.states[h - 1];
}
// DuplexModCodeRepr's derived order: Canonical < Code(char) < ChEbi(n)
__device__ __forceinline__ unsigned long long hemi_half_order(uint32_t code) {
    return code == 0 ? 0ull : (code & 0x80000000u) ? (1ull << 32) + (code & 0x7fffffffu) : 1ull + code;
}

__device__ uint32_t hemi_column_rows(const HemiRowDev& R, const uint32_t* S, uint32_t pos, mkp_hemi_row* out) {
    uint32_t mod_calls[4] = {0, 0, 0, 0};
    for (uint32_t id = 0; id < R.n_pat; id++) {
        const uint32_t v = S[HS_PAT + id], b = R.pat_keys[id] & 3u;
#pragma unroll
        for (uint32_t k = 0; k < 4; k++) if (k == b) mod_calls[k] += v;
    }
    uint32_t n = 0;
    for (uint32_t pb = 0; pb < 4; pb++) {
        if (!mod_calls[pb]) continue;
        uint32_t n_diff = 0, n_canon = 0;
        for (uint32_t b = 0; b < 4; b++) if (b != pb) n_diff += mod_calls[b];
        for (uint32_t id = 0; id < R.n_pat; id++) if (R.pat_keys[id] == hemi_key(pb, 0, 0)) n_canon = S[HS_PAT + id];
        const uint32_t row0 = n;
        for (uint32_t id = 0; id < R.n_pat; id++) {
            const uint32_t key = R.pat_keys[id], cnt = S[HS_PAT + id];
            if ((key & 3u) != pb || !cnt) continue;
            if (out) {
                // insertion sort of this base's rows by (top, bottom): shift the larger rows up, then write the fields in place
                const uint32_t tc = hemi_half_code(R, pb, (key >> 2) & 63u), bc = hemi_half_code(R, pb, (key >> 8) & 63u);
                const unsigned long long kt = hemi_half_order(tc), kb = hemi_half_order(bc);
                uint32_t j = n;
                while (j > row0) {
                    const unsigned long long pt = hemi_half_order(out[j - 1].top_code), pbo = hemi_half_order(out[j - 1].bottom_code);
                    if (pt < kt || (pt == kt && pbo < kb)) break;
                    out[j] = out[j - 1];
                    j--;
                }
                mkp_hemi_row* r = out + j;
                r->pos = pos; r->primary_base = (uint8_t)pb; r->reserved[0] = r->reserved[1] = r->reserved[2] = 0;
                r->top_code = tc; r->bottom_code = bc;
                r->count = cnt; r->n_canonical = n_canon; r->n_other_pattern = mod_calls[pb] - cnt;
                r->n_delete = S[HS_DEL]; r->n_fail = S[HS_FAIL + pb]; r->n_diff = n_diff; r->n_nocall = S[HS_NOCALL + pb];
            }
            n++;
        }
    }
    return n;
}

// thread per column word; EMIT = false counts the rows of the word, true writes them at row_prefix[w]
template <bool EMIT>
__global__ void __launch_bounds__(256) k_hemi_rows(HemiRowDev R) {
    const uint32_t w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= R.n_words) return;
    uint32_t bits = R.cols[w];
    if (!bits) { if (!EMIT) R.row_counts[w] = 0; return; }
    uint32_t slot = R.col_prefix[w];
    uint32_t n = 0;
    mkp_hemi_row* out = EMIT ? R.rows + R.row_prefix[w] : nullptr;
    while (bits) {
        const uint32_t bit = __ffs(bits) - 1;
        bits &= bits - 1;
        n += hemi_column_rows(R, R.slots + (size_t)slot * R.stride, R.cs + (w << 5) + bit, EMIT ? out + n : nullptr);
        slot++;
    }
    if (!EMIT) R.row_counts[w] = n;
}

}  // namespace mkp
