// C ABI (include/mkp.h) over the sm_100a kernels in mkp_kernels.cuh.
// One mkp_ctx per GPU: grow-only device buffers, one stream, CUDA events around every stage.
#include <cuda_runtime.h>
#include <atomic>
#include <unistd.h>
#include <chrono>
#include <sched.h>

#include <algorithm>
#include <cctype>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "mkp_kernels.cuh"
#include "mkp_fused.cuh"
#include "mkp_tile.cuh"
#include "mkp_ingest.cuh"
#include "mkp_hemi.cuh"

using namespace mkp;

namespace {

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        // slack: chunk buffers grow with the largest chunk seen so far; a quarter on top keeps the regrowth (free + malloc of
        // GB-sized buffers, a device synchronisation each) to one or two per run. The file / inflated-stream buffers get less.
        size_t want = bytes + (bytes < ((size_t)4 << 30) ? bytes / 4 : bytes / 8) + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return (T*)p; }
};

}  // namespace

struct mkp_ctx {
    int device = 0;
    cudaStream_t stream = nullptr, stream2 = nullptr;   // stream2: k_count_calls runs beside k_count_bases
    cudaEvent_t ev[10];
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    std::string err;
    mkp_params params;
    bool have_params = false;
    int sm_count = 148;
    // resident chunk
    DevBuf d_hdrs, d_heap, d_entry_off, d_focus_pos, d_focus_neg;
    uint32_t n_reads = 0, cs = 0, ce = 0, n_words = 0;
    bool have_focus = false;
    uint64_t total_entries = 0;
    uint32_t max_ncigar = 1, max_blocks = 1;
    uint64_t heap_bytes = 0;
    // work buffers
    DevBuf d_rl, d_meta, d_P, d_calls, d_hot, d_hot_prefix, d_block_sums, d_small, d_scr_cq, d_scr_cr, d_slow;
    DevBuf d_obs_word, d_slots, d_row_counts, d_row_prefix, d_rows, d_hist, d_take;
    // device ingest (BGZF file, inflated BAM stream, record table, slicing scratch)
    DevBuf d_file, d_members, d_bam, d_seeds, d_seg_counts, d_seg_base, d_recs, d_ids, d_plan, d_need, d_totals, d_slab_work;
    uint64_t bam_len = 0;
    size_t n_records = 0;
    bool inflate_attr_set = false;
    // results
    size_t n_rows = 0;
    uint64_t launches = 0;       // kernels launched by this context (mkp_kernel_launches)
    double pass_prof[4] = {0, 0, 0, 0};          // same for the pileup pass: buffers, launches, wait, calls
    double slice_prof[6] = {0, 0, 0, 0, 0, 0};   // MKP_TRACE_SLICE=1: host seconds in the phases of mkp_bam_chunk, printed by mkp_destroy
    // fused pass (chunks with focus bitmaps): tile table, rank of the focus set (built at upload), capacities
    DevBuf d_pscr, d_inftab, d_tiles, d_order;
    bool order_ready = false;
    uint32_t n_tiles = 0;
    bool tile_attr_set = false;
    uint32_t n_hot = 0, state_cap = 4, p_stride = 0;
    bool fused_attr_set = false, focus_ready = false;
    // pinned staging buffers for host -> device copies of pageable memory (the mapped BAM file): one per copy thread
    static constexpr int N_PIN = 16;                       // staging buffers allocated (MKP_H2D_THREADS of them are used, default 6)
    static constexpr size_t PIN_BYTES = (size_t)16 << 20;
    void* pin[N_PIN] = {};
    int n_pin = 0;
    cudaEvent_t pin_ev[N_PIN];
    bool pin_ready = false;
    std::vector<mkp_row> h_rows;
    std::vector<uint64_t> h_entry_off;
    mkp_row* h_rows_pinned = nullptr;
    size_t h_rows_pinned_cap = 0;
    // pileup-hemi: pattern registry, interval starts, column rank, per-column counters, rows
    DevBuf d_hemi_pat, d_hemi_iv, d_hemi_prefix, d_hemi_slots, d_hemi_rows;
    uint32_t hemi_pat_cap = 8;
    size_t n_hemi_rows = 0;
    std::vector<mkp_hemi_row> h_hemi_rows;
};

static_assert(sizeof(mkp_hemi_row) == 44, "mkp_hemi_row is part of the C ABI");

// d_small layout (u64 words): [0..31] states, [32] total_calls, [33] hist_inexact ; u32 view from byte 34*8: n_states, err, n_hot, n_rows
static constexpr size_t SMALL_BYTES = 34 * 8 + 16 * 4;

static int fail(mkp_ctx* c, const std::string& m, int code = -1) { if (c) c->err = m; return code; }
#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(ctx, std::string(#call) + ": " + cudaGetErrorString(e_)); } while (0)

extern "C" {

static int finish_upload(mkp_ctx* ctx);

int mkp_create(int device, mkp_ctx** out) {
    if (!out) return -1;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) return -2;   // no CUDA device: there is no CPU fallback
    if (device < 0 || device >= n) return -3;
    if (cudaSetDevice(device) != cudaSuccess) return -4;
    mkp_ctx* ctx = new mkp_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) ctx->sm_count = prop.multiProcessorCount;
    if (cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return -5; }
    if (cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking) != cudaSuccess) { delete ctx; return -5; }
    for (auto& e : ctx->ev) cudaEventCreate(&e);
    cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming);
    cudaEventCreateWithFlags(&ctx->ev_join, cudaEventDisableTiming);
    memset(&ctx->params, 0, sizeof ctx->params);
    *out = ctx;
    return 0;
}

int mkp_bind_host_thread(int device) {
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) return -1;
    for (char* c = bus; *c; c++) *c = (char)tolower((unsigned char)*c);
    char path[128];
    snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
    FILE* f = fopen(path, "r");
    if (!f) return 1;
    int node = -1;
    const int got = fscanf(f, "%d", &node);
    fclose(f);
    if (got != 1 || node < 0) return 1;
    snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
    f = fopen(path, "r");
    if (!f) return 1;
    char list[4096] = {0};
    const size_t n = fread(list, 1, sizeof list - 1, f);
    fclose(f);
    if (!n) return 1;
    cpu_set_t set;
    CPU_ZERO(&set);
    int any = 0;
    for (char* p = list; *p;) {           // "0-31,64-95"
        char* e;
        long a = strtol(p, &e, 10);
        if (e == p) break;
        long b = a;
        if (*e == '-') { p = e + 1; b = strtol(p, &e, 10); }
        for (long c = a; c <= b && c < CPU_SETSIZE; c++) { CPU_SET((int)c, &set); any = 1; }
        p = e;
        while (*p == ',' || *p == '\n' || *p == ' ') p++;
    }
    if (!any) return 1;
    return sched_setaffinity(0, sizeof set, &set) == 0 ? 0 : -2;
}

void mkp_destroy(mkp_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (getenv("MKP_TRACE_SLICE")) fprintf(stderr, "[mkp] slice phases (s): buffers %.4f plan+scan %.4f heap alloc %.4f copy+focus %.4f finish_upload %.4f calls %.0f\n",
                                           ctx->slice_prof[0], ctx->slice_prof[1], ctx->slice_prof[2], ctx->slice_prof[3], ctx->slice_prof[4], ctx->slice_prof[5]);
    if (getenv("MKP_TRACE_SLICE")) fprintf(stderr, "[mkp] pass phases (s): buffers %.4f launches %.4f wait %.4f calls %.0f\n", ctx->pass_prof[0], ctx->pass_prof[1], ctx->pass_prof[2], ctx->pass_prof[3]);
    DevBuf* bufs[] = {&ctx->d_hdrs, &ctx->d_heap, &ctx->d_entry_off, &ctx->d_focus_pos, &ctx->d_focus_neg, &ctx->d_rl, &ctx->d_meta, &ctx->d_P,
                      &ctx->d_calls, &ctx->d_hot, &ctx->d_hot_prefix, &ctx->d_block_sums, &ctx->d_small, &ctx->d_scr_cq, &ctx->d_scr_cr, &ctx->d_slow,
                      &ctx->d_obs_word, &ctx->d_slots, &ctx->d_row_counts, &ctx->d_row_prefix, &ctx->d_rows, &ctx->d_hist, &ctx->d_take,
                      &ctx->d_file, &ctx->d_members, &ctx->d_bam, &ctx->d_seeds, &ctx->d_seg_counts, &ctx->d_seg_base, &ctx->d_recs, &ctx->d_ids, &ctx->d_plan,
                      &ctx->d_need, &ctx->d_totals, &ctx->d_slab_work, &ctx->d_pscr, &ctx->d_inftab, &ctx->d_tiles, &ctx->d_order,
                      &ctx->d_hemi_pat, &ctx->d_hemi_iv, &ctx->d_hemi_prefix, &ctx->d_hemi_slots, &ctx->d_hemi_rows};
    for (auto* b : bufs) b->release();
    if (ctx->h_rows_pinned) cudaFreeHost(ctx->h_rows_pinned);
    for (int i = 0; i < ctx->n_pin; i++) { cudaFreeHost(ctx->pin[i]); cudaEventDestroy(ctx->pin_ev[i]); }
    for (auto& e : ctx->ev) cudaEventDestroy(e);
    cudaEventDestroy(ctx->ev_fork); cudaEventDestroy(ctx->ev_join);
    cudaStreamDestroy(ctx->stream2);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* mkp_last_error(const mkp_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int mkp_set_params(mkp_ctx* ctx, const mkp_params* p) {
    if (!ctx || !p) return -1;
    if (p->n_mod_thresholds > MKP_MAX_MOD_THRESHOLDS) return fail(ctx, "too many per-mod thresholds");
    CK(cudaSetDevice(ctx->device));
    ctx->params = *p;
    DevParams d;
    memset(&d, 0, sizeof d);
    d.default_thr = p->default_threshold;
    for (int b = 0; b < 4; b++) { d.base_thr[b] = p->base_threshold[b]; d.base_set[b] = p->base_threshold_set[b] ? 1 : 0; }
    d.n_mod_thr = p->n_mod_thresholds;
    for (uint32_t i = 0; i < p->n_mod_thresholds; i++) { d.mod_code[i] = p->mod_code[i]; d.mod_thr[i] = p->mod_threshold[i]; }
    d.numeric_mode = p->numeric_mode; d.collapse_code = p->collapse_code; d.force_allow_implicit = p->force_allow_implicit;
    d.edge_on = p->edge_filter_on; d.edge_inv = p->edge_filter_inverted; d.edge_start = p->edge_filter_start; d.edge_end = p->edge_filter_end;
    CK(cudaMemcpyToSymbolAsync(c_par, &d, sizeof d, 0, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->have_params = true;
    return 0;
}

int mkp_upload_chunk(mkp_ctx* ctx, const mkp_chunk* ch) {
    if (!ctx || !ch) return -1;
    if (ch->end <= ch->start) return fail(ctx, "empty chunk range");
    CK(cudaSetDevice(ctx->device));
    ctx->n_reads = ch->n_reads; ctx->cs = ch->start; ctx->ce = ch->end;
    ctx->n_words = (ch->end - ch->start + 31) / 32;
    ctx->heap_bytes = ch->heap_bytes;
    ctx->h_entry_off.resize((size_t)ch->n_reads + 1);
    uint64_t acc = 0;
    uint32_t mc = 1, ml = 1;
    for (uint32_t i = 0; i < ch->n_reads; i++) {
        ctx->h_entry_off[i] = acc;
        acc += ch->hdrs[i].len_ml;
        mc = std::max(mc, ch->hdrs[i].n_cigar);
        ml = std::max(ml, ch->hdrs[i].l_seq);
    }
    ctx->h_entry_off[ch->n_reads] = acc;
    ctx->total_entries = acc;
    ctx->max_ncigar = mc;
    ctx->max_blocks = (ml + 31) / 32;
    CK(ctx->d_hdrs.ensure(std::max<size_t>(1, ch->n_reads) * sizeof(mkp_read_hdr)));
    CK(ctx->d_heap.ensure(ch->heap_bytes + 64));
    CK(ctx->d_entry_off.ensure(((size_t)ch->n_reads + 1) * 8));
    if (ch->n_reads) {
        CK(cudaMemcpyAsync(ctx->d_hdrs.p, ch->hdrs, (size_t)ch->n_reads * sizeof(mkp_read_hdr), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_heap.p, ch->heap, ch->heap_bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    CK(cudaMemcpyAsync(ctx->d_entry_off.p, ctx->h_entry_off.data(), ((size_t)ch->n_reads + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    ctx->have_focus = ch->focus_pos && ch->focus_neg;
    if (ctx->have_focus) {
        CK(ctx->d_focus_pos.ensure((size_t)ctx->n_words * 4));
        CK(ctx->d_focus_neg.ensure((size_t)ctx->n_words * 4));
        CK(cudaMemcpyAsync(ctx->d_focus_pos.p, ch->focus_pos, (size_t)ctx->n_words * 4, cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_focus_neg.p, ch->focus_neg, (size_t)ctx->n_words * 4, cudaMemcpyHostToDevice, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return finish_upload(ctx);
}

static int decode_grid(const mkp_ctx* ctx, uint32_t n_reads) {
    int blocks = ctx->sm_count * 12;                   // 48 warps per SM at 4 warps per block
    int need = (int)((n_reads + 3) / 4);
    return std::max(1, std::min(blocks, need));
}

static int prepare_decode(mkp_ctx* ctx, ChunkDev* C, int grid) {
    const size_t nwarps = (size_t)grid * 4;
    CK(ctx->d_meta.ensure(std::max<size_t>(1, ctx->n_reads) * sizeof(ReadMeta)));
    CK(ctx->d_rl.ensure(std::max<size_t>(1, ctx->n_reads) * sizeof(ReadLists)));
    CK(ctx->d_P.ensure(std::max<uint64_t>(1, ctx->total_entries) * 4));
    CK(ctx->d_calls.ensure(std::max<uint64_t>(1, ctx->total_entries) * 8));
    CK(ctx->d_hot.ensure((size_t)ctx->n_words * 4 + 4));
    CK(ctx->d_hot_prefix.ensure((size_t)ctx->n_words * 4 + 4));
    CK(ctx->d_small.ensure(SMALL_BYTES));
    CK(ctx->d_scr_cq.ensure(nwarps * ((size_t)ctx->max_ncigar + 4) * 4));
    CK(ctx->d_scr_cr.ensure(nwarps * ((size_t)ctx->max_ncigar + 4) * 4));
    memset(C, 0, sizeof *C);
    C->hdrs = ctx->d_hdrs.as<mkp_read_hdr>(); C->heap = ctx->d_heap.as<uint8_t>(); C->entry_off = ctx->d_entry_off.as<uint64_t>();
    C->n_reads = ctx->n_reads; C->cs = ctx->cs; C->ce = ctx->ce;
    C->focus_pos = ctx->have_focus ? ctx->d_focus_pos.as<uint32_t>() : nullptr;
    C->focus_neg = ctx->have_focus ? ctx->d_focus_neg.as<uint32_t>() : nullptr;
    C->meta = ctx->d_meta.as<ReadMeta>(); C->P = ctx->d_P.as<uint32_t>(); C->calls = ctx->d_calls.as<uint2>();
    C->hot = ctx->d_hot.as<uint32_t>(); C->hot_prefix = ctx->d_hot_prefix.as<uint32_t>();
    C->states = ctx->d_small.as<unsigned long long>();
    C->total_calls = C->states + 32;
    C->hist_inexact = C->states + 33;
    uint32_t* u = (uint32_t*)(ctx->d_small.as<uint8_t>() + 34 * 8);
    C->n_states = u; C->err = u + 1; C->work = u + 4;
    C->scr_cq = ctx->d_scr_cq.as<uint32_t>(); C->scr_cr = ctx->d_scr_cr.as<uint32_t>();
    C->max_ncigar = ctx->max_ncigar; C->max_blocks = ctx->max_blocks;
    C->rl = ctx->d_rl.as<ReadLists>();
    CK(ctx->d_slow.ensure((size_t)ctx->n_reads * 4 + 4));
    C->slow_list = ctx->d_slow.as<uint32_t>();
    C->order = ctx->order_ready ? ctx->d_order.as<uint32_t>() : nullptr;
    return 0;
}

static std::string derr_text(uint32_t e) {
    std::string s;
    if (e & MKP_DERR_TOO_MANY_STATES) s += "more than 32 distinct (base, mod code) states; ";
    if (e & MKP_DERR_TOO_MANY_LISTS) s += "more than 16 MM lists in one read; ";
    if (e & MKP_DERR_TOO_MANY_CODES) s += "more than 4 codes in one MM list or 7 at one position; ";
    if (e & MKP_DERR_TOO_MANY_PATTERNS) s += "more than 256 distinct (base, top, bottom) hemi patterns in one chunk; ";
    return s;
}

// Chunks with focus bitmaps: the positions that can produce rows are known at upload, so the rank structure (counter slot of
// every focus position) and the tile table of the fused pass are built here, once per chunk, not once per pass.
static int finish_upload(mkp_ctx* ctx) {
    ctx->focus_ready = false;
    ctx->order_ready = false;
    cudaStream_t st = ctx->stream;
    if (ctx->n_reads >= 4096 && !getenv("MKP_NO_ORDER")) {            // processing order of the read queues: longest reads first
        CK(ctx->d_order.ensure((size_t)ctx->n_reads * 4 + 32 * 4));
        uint32_t* hist = ctx->d_order.as<uint32_t>() + ctx->n_reads;
        CK(cudaMemsetAsync(hist, 0, 32 * 4, st));
        const int g = (int)((ctx->n_reads + 255) / 256);
        ctx->launches += 3;
        k_order_hist<<<g, 256, 0, st>>>(ctx->d_hdrs.as<mkp_read_hdr>(), ctx->n_reads, hist);
        k_order_scan<<<1, 1, 0, st>>>(hist);
        k_order_scatter<<<g, 256, 0, st>>>(ctx->d_hdrs.as<mkp_read_hdr>(), ctx->n_reads, hist, ctx->d_order.as<uint32_t>());
        ctx->order_ready = true;
    }
    if (!ctx->have_focus) { CK(cudaStreamSynchronize(st)); CK(cudaGetLastError()); return 0; }
    const uint32_t n_words = ctx->n_words;
    const uint32_t n_blk = (n_words + 1023) / 1024;
    CK(ctx->d_hot.ensure((size_t)n_words * 4 + 4));
    CK(ctx->d_hot_prefix.ensure((size_t)n_words * 4 + 4));
    CK(ctx->d_block_sums.ensure((size_t)n_blk * 4 + 4));
    CK(ctx->d_small.ensure(SMALL_BYTES));
    uint32_t* u = (uint32_t*)(ctx->d_small.as<uint8_t>() + 34 * 8);
    ctx->launches += 4;
    k_focus_union<<<(n_words + 255) / 256, 256, 0, st>>>(ctx->d_focus_pos.as<uint32_t>(), ctx->d_focus_neg.as<uint32_t>(), ctx->d_hot.as<uint32_t>(), n_words);
    k_block_popc<<<n_blk, 1024, 0, st>>>(ctx->d_hot.as<uint32_t>(), n_words, ctx->d_block_sums.as<uint32_t>(), nullptr, nullptr);
    k_scan_blocks<<<1, 1024, 0, st>>>(ctx->d_block_sums.as<uint32_t>(), n_blk, u + 2);
    k_word_prefix<<<n_blk, 1024, 0, st>>>(ctx->d_hot.as<uint32_t>(), n_words, ctx->d_block_sums.as<uint32_t>(), ctx->d_hot_prefix.as<uint32_t>());
    uint32_t n_hot = 0;
    CK(cudaMemcpyAsync(&n_hot, u + 2, 4, cudaMemcpyDeviceToHost, st));
    ctx->n_tiles = ctx->n_reads ? (uint32_t)((ctx->heap_bytes + TL_WIN - 1) / TL_WIN) : 0;
    if (ctx->n_tiles == 0 && ctx->n_reads) ctx->n_tiles = 1;
    CK(ctx->d_tiles.ensure(((size_t)ctx->n_tiles + 1) * sizeof(TileInfo)));
    ctx->launches += 1;
    k_tiles<<<(ctx->n_tiles + 1 + 255) / 256, 256, 0, st>>>(ctx->d_hdrs.as<mkp_read_hdr>(), ctx->n_reads, ctx->heap_bytes, ctx->d_tiles.as<TileInfo>(), ctx->n_tiles);
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    ctx->n_hot = n_hot;
    ctx->focus_ready = true;
    return 0;
}

// The pass for chunks with focus bitmaps: k_pileup_fused, the generic kernels over the reads it left, the row kernels. Everything
// is enqueued at once; the host reads the counters once, at the end (capacities that turn out too small - distinct
// (base, code) states per slot, rows - grow and the affected part runs again).
static int pileup_fused(mkp_ctx* ctx, mkp_stats* stats) {
    cudaStream_t st = ctx->stream;
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto since = [&](std::chrono::steady_clock::time_point t) { return std::chrono::duration<double>(now() - t).count(); };
    auto tp = now();
    const uint32_t n_words = ctx->n_words, n_hot = ctx->n_hot;
    const uint32_t n_blk = (n_words + 1023) / 1024;
    ChunkDev C;
    // MKP_FUSED=1: the TMA-staged single-traversal kernel (k_pileup_fused); default: the per-stage kernels (see DESIGN.md 4:
    // the pass is bound by instruction issue, and the per-stage kernels keep 2-3x more warps per SM in flight)
    const char* fz = getenv("MKP_FUSED");
    const char* tl = getenv("MKP_TILE");
    const bool use_tile = tl && tl[0] == '1';                  // k_pileup_tile: CTA-cooperative phases over TMA-staged tiles
    const bool use_fused = use_tile || (fz && fz[0] == '1');
    const int g_slow = use_fused ? std::max(1, std::min(ctx->sm_count * 2, (int)((ctx->n_reads + 3) / 4))) : decode_grid(ctx, ctx->n_reads);
    if (int rc = prepare_decode(ctx, &C, g_slow)) return rc;
    CK(ctx->d_block_sums.ensure((size_t)n_blk * 4 + 4));
    CK(ctx->d_row_counts.ensure((size_t)n_words * 4 + 4));
    CK(ctx->d_row_prefix.ensure((size_t)n_words * 4 + 4));
    CK(ctx->d_obs_word.ensure((size_t)n_words * 8 + 8));
    const int grid = ctx->sm_count;
    ctx->p_stride = std::min<uint32_t>(65536u, std::max<uint32_t>(1024u, 2u * ctx->max_blocks * 32u));
    CK(ctx->d_pscr.ensure((size_t)grid * FZ_WARPS * ctx->p_stride * 4));
    if (!ctx->fused_attr_set) {
        CK(cudaFuncSetAttribute(k_pileup_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(FzShared)));
        ctx->fused_attr_set = true;
    }
    uint32_t* u = (uint32_t*)(ctx->d_small.as<uint8_t>() + 34 * 8);   // n_states, err, n_hot, n_rows, work[0..5] = u+4.., tile counter u+12
    uint32_t h_small[4] = {0, 0, 0, 0};
    unsigned long long h_calls = 0;
    uint32_t h_slow = 0;
    bool fused_ran = false;
    for (int attempt = 0;; attempt++) {
        const uint32_t S_cap = ctx->state_cap;
        const uint32_t stride = SL_MOD + 2 * S_cap;
        CK(ctx->d_slots.ensure(std::max<size_t>(1, n_hot) * stride * 4));
        if (!ctx->d_rows.p) CK(ctx->d_rows.ensure(std::max<size_t>(1024, (size_t)n_hot * 3) * sizeof(mkp_row)));
        ctx->pass_prof[0] += since(tp); tp = now();
        CK(cudaEventRecord(ctx->ev[0], st));
        CK(cudaMemsetAsync(ctx->d_small.p, 0xff, 32 * 8, st));
        CK(cudaMemsetAsync(ctx->d_small.as<uint8_t>() + 32 * 8, 0, SMALL_BYTES - 32 * 8, st));
        CK(cudaMemsetAsync(ctx->d_slots.p, 0, (size_t)n_hot * stride * 4, st));
        CK(cudaMemsetAsync(ctx->d_obs_word.p, 0, (size_t)n_words * 8, st));
        FusedDev F;
        memset(&F, 0, sizeof F);
        F.hdrs = C.hdrs; F.heap = C.heap; F.n_reads = C.n_reads; F.cs = C.cs; F.ce = C.ce;
        F.read_counter = u + 12;
        F.focus_pos = C.focus_pos; F.focus_neg = C.focus_neg; F.hot = C.hot; F.hot_prefix = C.hot_prefix;
        F.slots = ctx->d_slots.as<uint32_t>(); F.stride = stride; F.n_states = S_cap; F.n_words = n_words;
        F.obs_word = ctx->d_obs_word.as<uint32_t>();
        F.states = C.states; F.n_states_seen = C.n_states; F.err = C.err;
        F.slow_list = C.slow_list; F.slow_count = C.work + 4; F.total_calls = C.total_calls;
        F.p_scratch = ctx->d_pscr.as<uint32_t>(); F.p_stride = ctx->p_stride;
        C.mode = MODE_PILEUP;
        CountDev D;
        D.hdrs = C.hdrs; D.heap = C.heap; D.meta = C.meta; D.calls = C.calls; D.n_reads = C.n_reads; D.cs = C.cs; D.ce = C.ce;
        D.focus_pos = C.focus_pos; D.focus_neg = C.focus_neg; D.hot = C.hot; D.hot_prefix = C.hot_prefix;
        D.slots = F.slots; D.stride = stride; D.n_states = S_cap; D.n_words = n_words; D.obs_word = F.obs_word; D.work = u + 6;
        D.order = nullptr;          // (the counting kernels keep the coordinate order: neighbouring reads update neighbouring slots)
        if (use_fused) {
            if (ctx->n_reads && use_tile) {
                if (!ctx->tile_attr_set) { CK(cudaFuncSetAttribute(k_pileup_tile, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(TlShared))); ctx->tile_attr_set = true; }
                TileDev Tl;
                Tl.F = F; Tl.tiles = ctx->d_tiles.as<TileInfo>(); Tl.n_tiles = ctx->n_tiles; Tl.tile_counter = u + 13;
                ctx->launches += 1;
                k_pileup_tile<<<grid, TL_THREADS, sizeof(TlShared), st>>>(Tl);
            } else if (ctx->n_reads) { ctx->launches += 1; k_pileup_fused<<<grid, FZ_THREADS, sizeof(FzShared), st>>>(F); }
            CK(cudaEventRecord(ctx->ev[1], st));
            // the reads the fused kernel left to the generic path (list mode); both add into the same slots
            C.list_mode = 1;
            D.list = C.slow_list; D.list_count = C.work + 4;
            if (ctx->n_reads) {
                ctx->launches += 4;
                k_parse<<<g_slow, 128, 0, st>>>(C);
                k_resolve<MODE_PILEUP, false><<<g_slow, 128, 0, st>>>(C);
                const int g2 = std::max(1, std::min(ctx->sm_count * 2, (int)((ctx->n_reads + 7) / 8)));
                k_count_calls<<<g2, 256, 0, st>>>(D);
                k_count_bases<<<g2, 256, 0, st>>>(D);
            }
            CK(cudaEventRecord(ctx->ev[2], st));
            CK(cudaEventRecord(ctx->ev[4], st));
        } else {
            // the per-stage kernels at full occupancy (every read), counters addressed by the rank of the focus bit: no hot
            // marks, no rank pass, no host round trip between the stages
            C.list_mode = 2;
            D.list = nullptr; D.list_count = nullptr;
            const int gd = decode_grid(ctx, ctx->n_reads);
            if (ctx->n_reads) {
                ctx->launches += 5;
                k_parse<<<gd, 128, 0, st>>>(C);
                CK(cudaEventRecord(ctx->ev[1], st));
                k_resolve<MODE_PILEUP, true><<<gd, 128, 0, st>>>(C);
                k_resolve<MODE_PILEUP, false><<<gd, 128, 0, st>>>(C);
                CK(cudaEventRecord(ctx->ev[2], st));
                const int g2 = std::max(1, std::min(ctx->sm_count * 8, (int)((ctx->n_reads + 7) / 8)));
                CK(cudaEventRecord(ctx->ev_fork, st));
                CK(cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
                k_count_calls<<<g2, 256, 0, ctx->stream2>>>(D);
                CK(cudaEventRecord(ctx->ev_join, ctx->stream2));
                k_count_bases<<<g2, 256, 0, st>>>(D);
                CK(cudaStreamWaitEvent(st, ctx->ev_join, 0));
            } else { CK(cudaEventRecord(ctx->ev[1], st)); CK(cudaEventRecord(ctx->ev[2], st)); }
            CK(cudaEventRecord(ctx->ev[4], st));
        }
        RowDev R;
        R.hot = C.hot; R.hot_prefix = C.hot_prefix; R.n_words = n_words; R.cs = C.cs; R.ce = C.ce;
        R.slots = F.slots; R.stride = stride; R.n_states = S_cap; R.states = C.states; R.numeric_mode = ctx->params.numeric_mode;
        R.obs_word = F.obs_word;
        R.row_counts = ctx->d_row_counts.as<uint32_t>(); R.row_prefix = ctx->d_row_prefix.as<uint32_t>();
        R.rows = ctx->d_rows.as<mkp_row>(); R.rows_cap = (uint32_t)std::min<size_t>(0xffffffffu, ctx->d_rows.cap / sizeof(mkp_row));
        const int rg = (n_words + 255) / 256;
        ctx->launches += 5;
        k_rows<false><<<rg, 256, 0, st>>>(R);
        k_block_sum<<<n_blk, 1024, 0, st>>>(R.row_counts, n_words, ctx->d_block_sums.as<uint32_t>());
        k_scan_blocks<<<1, 1024, 0, st>>>(ctx->d_block_sums.as<uint32_t>(), n_blk, u + 3);
        k_value_prefix<<<n_blk, 1024, 0, st>>>(R.row_counts, n_words, ctx->d_block_sums.as<uint32_t>(), ctx->d_row_prefix.as<uint32_t>());
        k_rows<true><<<rg, 256, 0, st>>>(R);
        CK(cudaEventRecord(ctx->ev[3], st));
        fused_ran = use_fused;
        CK(cudaMemcpyAsync(h_small, u, 16, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&h_slow, u + 8, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&h_calls, C.total_calls, 8, cudaMemcpyDeviceToHost, st));
        ctx->pass_prof[1] += since(tp); tp = now();
        CK(cudaStreamSynchronize(st));
        CK(cudaGetLastError());
        ctx->pass_prof[2] += since(tp); tp = now();
        if (h_small[1]) {
            if (stats) { memset(stats, 0, sizeof *stats); stats->device_error = h_small[1]; }
            return fail(ctx, "device decode error: " + derr_text(h_small[1]), -10);
        }
        if (h_small[0] > S_cap) {                       // more distinct states than the slot layout holds: widen it, run again
            uint32_t c = S_cap;
            while (c < h_small[0]) c *= 2;
            ctx->state_cap = std::min<uint32_t>(c, MAX_STATES);
            if (attempt > 4) return fail(ctx, "state capacity did not converge");
            continue;
        }
        if (h_small[3] > R.rows_cap) {                  // more rows than the buffer holds: grow it, emit again
            CK(ctx->d_rows.ensure((size_t)h_small[3] * sizeof(mkp_row)));
            R.rows = ctx->d_rows.as<mkp_row>(); R.rows_cap = (uint32_t)std::min<size_t>(0xffffffffu, ctx->d_rows.cap / sizeof(mkp_row));
            ctx->launches += 1;
            k_rows<true><<<rg, 256, 0, st>>>(R);
            CK(cudaEventRecord(ctx->ev[3], st));
            CK(cudaStreamSynchronize(st));
            CK(cudaGetLastError());
        }
        break;
    }
    ctx->n_rows = h_small[3];
    ctx->pass_prof[3] += 1;
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->n_rows = h_small[3]; stats->n_hot = n_hot; stats->n_calls = h_calls; stats->n_states = h_small[0];
        stats->n_reads_skipped = h_slow;            // reads that went through the generic kernels
        auto el = [&](int a, int b) { float ms = 0; cudaEventElapsedTime(&ms, ctx->ev[a], ctx->ev[b]); return ms; };
        // kernel_ms: 0 parse (fused: the fused pass), incl. the clearing of the slots; 1 resolve (fused: generic kernels over the listed
        // reads); 4 counters; 5 rows; 6 host syncs (none on this path); 7 total
        stats->kernel_ms[0] = el(0, 1); stats->kernel_ms[1] = el(1, 2); stats->kernel_ms[4] = el(2, 4); stats->kernel_ms[5] = el(4, 3); stats->kernel_ms[7] = el(0, 3);
        if (!fused_ran) stats->n_reads_skipped = 0;
    }
    return 0;
}

int mkp_pileup_resident(mkp_ctx* ctx, mkp_stats* stats) {
    if (!ctx) return -1;
    if (!ctx->have_params) return fail(ctx, "mkp_set_params was not called");
    if (ctx->ce <= ctx->cs) return fail(ctx, "no resident chunk");
    CK(cudaSetDevice(ctx->device));
    if (ctx->have_focus && ctx->focus_ready && !getenv("MKP_NO_FOCUS_RANK")) return pileup_fused(ctx, stats);
    cudaStream_t st = ctx->stream;
    ChunkDev C;
    const int grid = decode_grid(ctx, ctx->n_reads);
    if (int rc = prepare_decode(ctx, &C, grid)) return rc;
    const uint32_t n_words = ctx->n_words;
    const uint32_t n_blk = (n_words + 1023) / 1024;
    CK(ctx->d_block_sums.ensure((size_t)n_blk * 4 + 4));
    CK(ctx->d_row_counts.ensure((size_t)n_words * 4 + 4));
    CK(ctx->d_row_prefix.ensure((size_t)n_words * 4 + 4));

    // events: 0 start | 1 after parse | 2 after resolve | 3 after rank | 4 before counts | 5 after count_calls |
    //         6 after count_bases | 7 after row count+scan | 8 before emit | 9 end
    CK(cudaEventRecord(ctx->ev[0], st));
    CK(cudaMemsetAsync(ctx->d_hot.p, 0, (size_t)n_words * 4, st));
    CK(cudaMemsetAsync(ctx->d_small.p, 0xff, 32 * 8, st));
    CK(cudaMemsetAsync(ctx->d_small.as<uint8_t>() + 32 * 8, 0, SMALL_BYTES - 32 * 8, st));
    C.mode = MODE_PILEUP;
    ctx->launches += 1; if (ctx->n_reads) k_parse<<<grid, 128, 0, st>>>(C);
    CK(cudaEventRecord(ctx->ev[1], st));
    ctx->launches += 2; if (ctx->n_reads) { k_resolve<MODE_PILEUP, true><<<grid, 128, 0, st>>>(C); k_resolve<MODE_PILEUP, false><<<grid, 128, 0, st>>>(C); }
    CK(cudaEventRecord(ctx->ev[2], st));
    uint32_t* u = (uint32_t*)(ctx->d_small.as<uint8_t>() + 34 * 8);   // n_states, err, n_hot, n_rows
    ctx->launches += 1; k_block_popc<<<n_blk, 1024, 0, st>>>(C.hot, n_words, ctx->d_block_sums.as<uint32_t>(), C.focus_pos, C.focus_neg);
    ctx->launches += 1; k_scan_blocks<<<1, 1024, 0, st>>>(ctx->d_block_sums.as<uint32_t>(), n_blk, u + 2);
    ctx->launches += 1; k_word_prefix<<<n_blk, 1024, 0, st>>>(C.hot, n_words, ctx->d_block_sums.as<uint32_t>(), C.hot_prefix);
    CK(cudaEventRecord(ctx->ev[3], st));
    uint32_t h_small[4];
    unsigned long long h_calls = 0;
    CK(cudaMemcpyAsync(h_small, u, 16, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&h_calls, C.total_calls, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const uint32_t n_states = h_small[0], derr = h_small[1], n_hot = h_small[2];
    if (derr) {
        if (stats) { memset(stats, 0, sizeof *stats); stats->device_error = derr; }
        return fail(ctx, "device decode error: " + derr_text(derr), -10);
    }
    const uint32_t stride = SL_MOD + 2 * std::max<uint32_t>(n_states, 1);
    CK(ctx->d_slots.ensure(std::max<size_t>(1, n_hot) * stride * 4));
    CK(cudaMemsetAsync(ctx->d_slots.p, 0, (size_t)n_hot * stride * 4, st));
    CK(ctx->d_obs_word.ensure((size_t)n_words * 8 + 8));
    CK(cudaMemsetAsync(ctx->d_obs_word.p, 0, (size_t)n_words * 8, st));
    CountDev D;
    D.hdrs = C.hdrs; D.heap = C.heap; D.meta = C.meta; D.calls = C.calls; D.n_reads = C.n_reads; D.cs = C.cs; D.ce = C.ce;
    D.focus_pos = C.focus_pos; D.focus_neg = C.focus_neg; D.hot = C.hot; D.hot_prefix = C.hot_prefix;
    D.slots = ctx->d_slots.as<uint32_t>(); D.stride = stride; D.n_states = std::max<uint32_t>(n_states, 1);
    D.n_words = n_words; D.obs_word = ctx->d_obs_word.as<uint32_t>(); D.work = u + 6;
    D.list = nullptr; D.list_count = nullptr; D.order = nullptr;      // (the counting kernels keep the coordinate order: neighbouring reads update neighbouring slots)
    CK(cudaEventRecord(ctx->ev[4], st));
    const int g2 = std::max(1, std::min(ctx->sm_count * 8, (int)((ctx->n_reads + 7) / 8)));
    // the two counting kernels only meet in commutative atomics on the slots: run them side by side (both are
    // latency-bound at 32 registers, so they co-reside on the SMs)
    CK(cudaEventRecord(ctx->ev_fork, st));
    CK(cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
    ctx->launches += 1; if (ctx->n_reads && n_hot) k_count_calls<<<g2, 256, 0, ctx->stream2>>>(D);
    CK(cudaEventRecord(ctx->ev_join, ctx->stream2));
    CK(cudaEventRecord(ctx->ev[5], st));
    ctx->launches += 1; if (ctx->n_reads && n_hot) k_count_bases<<<g2, 256, 0, st>>>(D);
    CK(cudaStreamWaitEvent(st, ctx->ev_join, 0));
    CK(cudaEventRecord(ctx->ev[6], st));
    RowDev R;
    R.hot = C.hot; R.hot_prefix = C.hot_prefix; R.n_words = n_words; R.cs = C.cs; R.ce = C.ce;
    R.slots = D.slots; R.stride = stride; R.n_states = D.n_states; R.states = C.states; R.numeric_mode = ctx->params.numeric_mode;
    R.obs_word = D.obs_word;
    R.row_counts = ctx->d_row_counts.as<uint32_t>(); R.row_prefix = ctx->d_row_prefix.as<uint32_t>(); R.rows = nullptr;
    const int rg = (n_words + 255) / 256;
    ctx->launches += 1; k_rows<false><<<rg, 256, 0, st>>>(R);
    ctx->launches += 1; k_block_sum<<<n_blk, 1024, 0, st>>>(R.row_counts, n_words, ctx->d_block_sums.as<uint32_t>());
    ctx->launches += 1; k_scan_blocks<<<1, 1024, 0, st>>>(ctx->d_block_sums.as<uint32_t>(), n_blk, u + 3);
    ctx->launches += 1; k_value_prefix<<<n_blk, 1024, 0, st>>>(R.row_counts, n_words, ctx->d_block_sums.as<uint32_t>(), ctx->d_row_prefix.as<uint32_t>());
    CK(cudaEventRecord(ctx->ev[7], st));
    uint32_t n_rows = 0;
    CK(cudaMemcpyAsync(&n_rows, u + 3, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(ctx->d_rows.ensure(std::max<size_t>(1, n_rows) * sizeof(mkp_row)));
    R.rows = ctx->d_rows.as<mkp_row>(); R.rows_cap = 0xffffffffu;
    CK(cudaEventRecord(ctx->ev[8], st));
    ctx->launches += 1; if (n_rows) k_rows<true><<<rg, 256, 0, st>>>(R);
    CK(cudaEventRecord(ctx->ev[9], st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    ctx->n_rows = n_rows;
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->n_rows = n_rows; stats->n_hot = n_hot; stats->n_calls = h_calls; stats->n_states = n_states;
        // kernel_ms: 0 parse, 1 resolve, 2 rank, 3 count_calls, 4 count_bases, 5 rows (count+scan+emit), 6 host syncs/allocs, 7 total
        auto el = [&](int a, int b) { float ms = 0; cudaEventElapsedTime(&ms, ctx->ev[a], ctx->ev[b]); return ms; };
        stats->kernel_ms[0] = el(0, 1); stats->kernel_ms[1] = el(1, 2); stats->kernel_ms[2] = el(2, 3);
        stats->kernel_ms[3] = 0.f; stats->kernel_ms[4] = el(4, 6);   // count_calls overlaps count_bases: [4] is the pair
        stats->kernel_ms[5] = el(6, 7) + el(8, 9);
        stats->kernel_ms[6] = el(3, 4) + el(7, 8); stats->kernel_ms[7] = el(0, 9);
    }
    return 0;
}

int mkp_fetch_rows(mkp_ctx* ctx, const mkp_row** rows, size_t* n_rows) {
    if (!ctx || !rows || !n_rows) return -1;
    CK(cudaSetDevice(ctx->device));
    if (ctx->n_rows > ctx->h_rows_pinned_cap) {
        if (ctx->h_rows_pinned) cudaFreeHost(ctx->h_rows_pinned);
        ctx->h_rows_pinned = nullptr; ctx->h_rows_pinned_cap = 0;
        size_t want = ctx->n_rows + ctx->n_rows / 8 + 1024;
        CK(cudaMallocHost((void**)&ctx->h_rows_pinned, want * sizeof(mkp_row)));
        ctx->h_rows_pinned_cap = want;
    }
    if (ctx->n_rows) {
        CK(cudaMemcpyAsync(ctx->h_rows_pinned, ctx->d_rows.p, ctx->n_rows * sizeof(mkp_row), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    *rows = ctx->h_rows_pinned;
    *n_rows = ctx->n_rows;
    return 0;
}

int mkp_pileup_chunk(mkp_ctx* ctx, const mkp_chunk* ch, const mkp_row** rows, size_t* n_rows, mkp_stats* stats) {
    if (int rc = mkp_upload_chunk(ctx, ch)) return rc;
    if (int rc = mkp_pileup_resident(ctx, stats)) return rc;
    return mkp_fetch_rows(ctx, rows, n_rows);
}

// `modkit pileup-hemi` on the resident chunk: the pileup decode (k_parse, k_resolve: every read's call records), the column rank,
// the pair kernel, the row kernels. The per-column counters hold `hemi_pat_cap` pattern counts; a chunk that shows more patterns
// grows the capacity and runs the pair kernel again (the decode stays).
int mkp_hemi_resident(mkp_ctx* ctx, int32_t offset, const uint32_t* interval_starts, uint32_t n_intervals, mkp_stats* stats) {
    if (!ctx) return -1;
    if (!ctx->have_params) return fail(ctx, "mkp_set_params was not called");
    if (ctx->ce <= ctx->cs) return fail(ctx, "no resident chunk");
    if (!ctx->have_focus) return fail(ctx, "mkp_hemi_resident needs the column / partner bitmaps (focus_pos / focus_neg)");
    if (!interval_starts || n_intervals == 0) return fail(ctx, "mkp_hemi_resident needs the interval starts of the chunk");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ChunkDev C;
    const int grid = decode_grid(ctx, ctx->n_reads);
    if (int rc = prepare_decode(ctx, &C, grid)) return rc;
    C.list_mode = 2;                                           // every read; the hot bitmap (rank of the focus set) is not touched
    const uint32_t n_words = ctx->n_words;
    const uint32_t n_blk = (n_words + 1023) / 1024;
    CK(ctx->d_block_sums.ensure((size_t)n_blk * 4 + 4));
    CK(ctx->d_row_counts.ensure((size_t)n_words * 4 + 4));
    CK(ctx->d_row_prefix.ensure((size_t)n_words * 4 + 4));
    CK(ctx->d_hemi_prefix.ensure((size_t)n_words * 4 + 4));
    CK(ctx->d_hemi_pat.ensure((HEMI_MAX_PATTERNS + 4) * 4));
    CK(ctx->d_hemi_iv.ensure((size_t)n_intervals * 4));
    uint32_t* pat = ctx->d_hemi_pat.as<uint32_t>();
    uint32_t* u = (uint32_t*)(ctx->d_small.as<uint8_t>() + 34 * 8);   // n_states, err, n_cols, n_rows; u[14] pair read counter
    // events: 0 start | 1 after parse | 2 after resolve | 3 after rank | 4 before pairs | 6 after pairs | 7 after row count+scan |
    //         8 before emit | 9 end
    CK(cudaEventRecord(ctx->ev[0], st));
    CK(cudaMemcpyAsync(ctx->d_hemi_iv.p, interval_starts, (size_t)n_intervals * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(pat, 0xff, HEMI_MAX_PATTERNS * 4, st));
    CK(cudaMemsetAsync(pat + HEMI_MAX_PATTERNS, 0, 16, st));
    CK(cudaMemsetAsync(ctx->d_small.p, 0xff, 32 * 8, st));
    CK(cudaMemsetAsync(ctx->d_small.as<uint8_t>() + 32 * 8, 0, SMALL_BYTES - 32 * 8, st));
    C.mode = MODE_PILEUP;
    ctx->launches += 1; if (ctx->n_reads) k_parse<<<grid, 128, 0, st>>>(C);
    CK(cudaEventRecord(ctx->ev[1], st));
    ctx->launches += 2; if (ctx->n_reads) { k_resolve<MODE_PILEUP, true><<<grid, 128, 0, st>>>(C); k_resolve<MODE_PILEUP, false><<<grid, 128, 0, st>>>(C); }
    CK(cudaEventRecord(ctx->ev[2], st));
    // counter slot of a column = rank of its bit in focus_pos
    uint32_t* cols = ctx->d_focus_pos.as<uint32_t>();
    uint32_t* col_prefix = ctx->d_hemi_prefix.as<uint32_t>();
    ctx->launches += 3;
    k_block_popc<<<n_blk, 1024, 0, st>>>(cols, n_words, ctx->d_block_sums.as<uint32_t>(), nullptr, nullptr);
    k_scan_blocks<<<1, 1024, 0, st>>>(ctx->d_block_sums.as<uint32_t>(), n_blk, u + 2);
    k_word_prefix<<<n_blk, 1024, 0, st>>>(cols, n_words, ctx->d_block_sums.as<uint32_t>(), col_prefix);
    CK(cudaEventRecord(ctx->ev[3], st));
    uint32_t h_small[4];
    unsigned long long h_calls = 0;
    CK(cudaMemcpyAsync(h_small, u, 16, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&h_calls, C.total_calls, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    const uint32_t n_states = h_small[0], derr = h_small[1], n_cols = h_small[2];
    if (derr) {
        if (stats) { memset(stats, 0, sizeof *stats); stats->device_error = derr; }
        return fail(ctx, "device decode error: " + derr_text(derr), -10);
    }
    HemiDev H;
    H.hdrs = C.hdrs; H.heap = C.heap; H.meta = C.meta; H.calls = C.calls; H.n_reads = C.n_reads; H.cs = C.cs; H.ce = C.ce;
    H.cols = cols; H.col_prefix = col_prefix; H.offset = offset;
    H.iv_starts = ctx->d_hemi_iv.as<uint32_t>(); H.n_iv = n_intervals;
    H.pat_keys = pat; H.n_pat = pat + HEMI_MAX_PATTERNS; H.work = u + 14;
    H.order = C.order; H.combine = ctx->params.numeric_mode == 1 ? 1u : 0u;
    const int g2 = std::max(1, std::min(ctx->sm_count * 8, (int)((ctx->n_reads + 7) / 8)));
    uint32_t n_pat = 0;
    float pairs_ms = 0;
    for (;;) {
        H.pat_cap = ctx->hemi_pat_cap;
        H.stride = HS_PAT + H.pat_cap;
        CK(ctx->d_hemi_slots.ensure(std::max<size_t>(1, n_cols) * H.stride * 4));
        H.slots = ctx->d_hemi_slots.as<uint32_t>();
        CK(cudaMemsetAsync(H.slots, 0, (size_t)n_cols * H.stride * 4, st));
        CK(cudaMemsetAsync(u + 14, 0, 4, st));
        CK(cudaEventRecord(ctx->ev[4], st));
        ctx->launches += 1; if (ctx->n_reads && n_cols) k_hemi_pairs<<<g2, 256, 0, st>>>(H);
        CK(cudaEventRecord(ctx->ev[6], st));
        CK(cudaMemcpyAsync(&n_pat, H.n_pat, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        float ms = 0;
        cudaEventElapsedTime(&ms, ctx->ev[4], ctx->ev[6]);
        pairs_ms += ms;
        if (n_pat > (uint32_t)HEMI_MAX_PATTERNS) {
            if (stats) { memset(stats, 0, sizeof *stats); stats->device_error = MKP_DERR_TOO_MANY_PATTERNS; }
            return fail(ctx, "device decode error: " + derr_text(MKP_DERR_TOO_MANY_PATTERNS), -10);
        }
        if (n_pat <= H.pat_cap) break;
        while (ctx->hemi_pat_cap < n_pat) ctx->hemi_pat_cap *= 2;     // more patterns than counters per column: grow, count again
    }
    HemiRowDev R;
    R.cols = cols; R.col_prefix = col_prefix; R.n_words = n_words; R.cs = C.cs;
    R.slots = H.slots; R.stride = H.stride; R.n_pat = n_pat; R.pat_keys = pat; R.states = C.states;
    R.row_counts = ctx->d_row_counts.as<uint32_t>(); R.row_prefix = ctx->d_row_prefix.as<uint32_t>(); R.rows = nullptr;
    const int rg = (n_words + 255) / 256;
    CK(cudaEventRecord(ctx->ev[6], st));
    ctx->launches += 4;
    k_hemi_rows<false><<<rg, 256, 0, st>>>(R);
    k_block_sum<<<n_blk, 1024, 0, st>>>(R.row_counts, n_words, ctx->d_block_sums.as<uint32_t>());
    k_scan_blocks<<<1, 1024, 0, st>>>(ctx->d_block_sums.as<uint32_t>(), n_blk, u + 3);
    k_value_prefix<<<n_blk, 1024, 0, st>>>(R.row_counts, n_words, ctx->d_block_sums.as<uint32_t>(), ctx->d_row_prefix.as<uint32_t>());
    CK(cudaEventRecord(ctx->ev[7], st));
    uint32_t n_rows = 0;
    CK(cudaMemcpyAsync(&n_rows, u + 3, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(ctx->d_hemi_rows.ensure(std::max<size_t>(1, n_rows) * sizeof(mkp_hemi_row)));
    R.rows = ctx->d_hemi_rows.as<mkp_hemi_row>();
    CK(cudaEventRecord(ctx->ev[8], st));
    ctx->launches += 1; if (n_rows) k_hemi_rows<true><<<rg, 256, 0, st>>>(R);
    CK(cudaEventRecord(ctx->ev[9], st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    ctx->n_hemi_rows = n_rows;
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->n_rows = n_rows; stats->n_hot = n_cols; stats->n_calls = h_calls; stats->n_states = n_states;
        auto el = [&](int a, int b) { float ms = 0; cudaEventElapsedTime(&ms, ctx->ev[a], ctx->ev[b]); return ms; };
        stats->kernel_ms[0] = el(0, 1); stats->kernel_ms[1] = el(1, 2); stats->kernel_ms[2] = el(2, 3);
        stats->kernel_ms[4] = pairs_ms; stats->kernel_ms[5] = el(6, 7) + el(8, 9);
        stats->kernel_ms[7] = el(0, 9); stats->kernel_ms[6] = stats->kernel_ms[7] - (el(0, 3) + pairs_ms + stats->kernel_ms[5]);
    }
    return 0;
}

int mkp_fetch_hemi_rows(mkp_ctx* ctx, const mkp_hemi_row** rows, size_t* n_rows) {
    if (!ctx || !rows || !n_rows) return -1;
    CK(cudaSetDevice(ctx->device));
    ctx->h_hemi_rows.resize(std::max<size_t>(1, ctx->n_hemi_rows));
    if (ctx->n_hemi_rows) {
        CK(cudaMemcpyAsync(ctx->h_hemi_rows.data(), ctx->d_hemi_rows.p, ctx->n_hemi_rows * sizeof(mkp_hemi_row), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    *rows = ctx->h_hemi_rows.data();
    *n_rows = ctx->n_hemi_rows;
    return 0;
}

int mkp_sample_histogram(mkp_ctx* ctx, int include_unaligned, const uint8_t* take, uint64_t* hist, uint8_t* contributes, uint64_t* inexact) {
    if (!ctx) return -1;
    if (!ctx->have_params) return fail(ctx, "mkp_set_params was not called");
    if (ctx->ce <= ctx->cs) return fail(ctx, "no resident chunk");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ChunkDev C;
    const int grid = decode_grid(ctx, ctx->n_reads);
    if (int rc = prepare_decode(ctx, &C, grid)) return rc;
    CK(cudaMemsetAsync(ctx->d_small.p, 0xff, 32 * 8, st));
    CK(cudaMemsetAsync(ctx->d_small.as<uint8_t>() + 32 * 8, 0, SMALL_BYTES - 32 * 8, st));
    C.hist_include_unaligned = include_unaligned ? 1 : 0;
    if (take) {
        CK(ctx->d_take.ensure(std::max<size_t>(1, ctx->n_reads)));
        CK(cudaMemcpyAsync(ctx->d_take.p, take, ctx->n_reads, cudaMemcpyHostToDevice, st));
        C.take = ctx->d_take.as<uint8_t>();
    }
    if (hist) {
        CK(ctx->d_hist.ensure(4 * 1025 * 8));
        CK(cudaMemsetAsync(ctx->d_hist.p, 0, 4 * 1025 * 8, st));
        C.hist = ctx->d_hist.as<unsigned long long>();
    }
    C.mode = MODE_HIST;
    ctx->launches += 3; if (ctx->n_reads) { k_parse<<<grid, 128, 0, st>>>(C); k_resolve<MODE_HIST, true><<<grid, 128, 0, st>>>(C); k_resolve<MODE_HIST, false><<<grid, 128, 0, st>>>(C); }
    CK(cudaGetLastError());
    uint32_t h_small[2];
    uint32_t* u = (uint32_t*)(ctx->d_small.as<uint8_t>() + 34 * 8);
    CK(cudaMemcpyAsync(h_small, u, 8, cudaMemcpyDeviceToHost, st));
    if (hist) CK(cudaMemcpyAsync(hist, ctx->d_hist.p, 4 * 1025 * 8, cudaMemcpyDeviceToHost, st));
    unsigned long long inx = 0;
    CK(cudaMemcpyAsync(&inx, C.hist_inexact, 8, cudaMemcpyDeviceToHost, st));
    std::vector<ReadMeta> metas;
    if (contributes) {
        metas.resize(ctx->n_reads);
        if (ctx->n_reads) CK(cudaMemcpyAsync(metas.data(), ctx->d_meta.p, (size_t)ctx->n_reads * sizeof(ReadMeta), cudaMemcpyDeviceToHost, st));
    }
    CK(cudaStreamSynchronize(st));
    if (h_small[1]) return fail(ctx, "device decode error: " + derr_text(h_small[1]), -10);
    if (contributes) for (uint32_t i = 0; i < ctx->n_reads; i++) contributes[i] = metas[i].n_hist > 0;
    if (inexact) *inexact = inx;
    return 0;
}


// `modkit summary` support: the calls of the reads flagged in `take`, classed with the thresholds of mkp_set_params
// (src/summarize.rs:117-252). Adds to table[4][2][33] (base, pass/fail, 0 canonical | 1 + state), reads_with[4], obs[4];
// states[32] receives the (base << 32 | code) key of every state id (~0 = unused).
int mkp_sample_summary(mkp_ctx* ctx, int include_unaligned, const uint8_t* take, uint64_t* table, uint64_t* reads_with, uint32_t* obs, uint64_t* states) {
    if (!ctx || !table || !reads_with || !obs || !states) return -1;
    if (!ctx->have_params) return fail(ctx, "mkp_set_params was not called");
    if (ctx->ce <= ctx->cs) return fail(ctx, "no resident chunk");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    ChunkDev C;
    const int grid = decode_grid(ctx, ctx->n_reads);
    if (int rc = prepare_decode(ctx, &C, grid)) return rc;
    CK(cudaMemsetAsync(ctx->d_small.p, 0xff, 32 * 8, st));
    CK(cudaMemsetAsync(ctx->d_small.as<uint8_t>() + 32 * 8, 0, SMALL_BYTES - 32 * 8, st));
    C.hist_include_unaligned = include_unaligned ? 1 : 0;
    if (take) {
        CK(ctx->d_take.ensure(std::max<size_t>(1, ctx->n_reads)));
        CK(cudaMemcpyAsync(ctx->d_take.p, take, ctx->n_reads, cudaMemcpyHostToDevice, st));
        C.take = ctx->d_take.as<uint8_t>();
    }
    const size_t words = 4 * 2 * 33 + 4 + 2;
    CK(ctx->d_hist.ensure(std::max<size_t>(4 * 1025, words) * 8));
    CK(cudaMemsetAsync(ctx->d_hist.p, 0, words * 8, st));
    C.summ = ctx->d_hist.as<unsigned long long>();
    C.mode = MODE_HIST;
    ctx->launches += 3;
    if (ctx->n_reads) { k_parse<<<grid, 128, 0, st>>>(C); k_resolve<MODE_HIST, true><<<grid, 128, 0, st>>>(C); k_resolve<MODE_HIST, false><<<grid, 128, 0, st>>>(C); }
    CK(cudaGetLastError());
    std::vector<uint64_t> h(words);
    uint32_t h_small[2];
    uint32_t* u = (uint32_t*)(ctx->d_small.as<uint8_t>() + 34 * 8);
    CK(cudaMemcpyAsync(h_small, u, 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(h.data(), ctx->d_hist.p, words * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(states, ctx->d_small.p, 32 * 8, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    if (h_small[1]) return fail(ctx, "device decode error: " + derr_text(h_small[1]), -10);
    for (int i = 0; i < 4 * 2 * 33; i++) table[i] += h[i];
    for (int b = 0; b < 4; b++) reads_with[b] += h[4 * 2 * 33 + b];
    const uint32_t* o32 = (const uint32_t*)(h.data() + 4 * 2 * 33 + 4);
    for (int b = 0; b < 4; b++) obs[b] = o32[b];
    return 0;
}

// ---- BGZF / BAM ingest on the device (mkp_ingest.cuh) -----------------------------------------------------
int mkp_device_memory(mkp_ctx* ctx, size_t* free_bytes, size_t* total_bytes) {
    if (!ctx) return -1;
    CK(cudaSetDevice(ctx->device));
    size_t f = 0, t = 0;
    CK(cudaMemGetInfo(&f, &t));
    if (free_bytes) *free_bytes = f;
    if (total_bytes) *total_bytes = t;
    return 0;
}

// Pageable host memory -> device at link speed: N_PIN host threads copy 16 MB pieces into their own pinned buffer and enqueue the
// transfer (a plain cudaMemcpyAsync from pageable memory is staged by the driver at ~10 GB/s). All transfers go to `st`.
// Source of a host -> device copy: bytes in memory, or - fd >= 0 - a file range read with pread() straight into the pinned staging
// buffers (no page of the file is mapped into the process: no page faults on the way in, nothing to unmap afterwards).
struct HostSrc { const uint8_t* mem; int fd; uint64_t fd_off; };
static bool read_fully(int fd, uint8_t* dst, size_t n, uint64_t off) {
    size_t got = 0;
    while (got < n) {
        const ssize_t r = pread(fd, dst + got, n - got, (off_t)(off + got));
        if (r <= 0) return false;
        got += (size_t)r;
    }
    return true;
}
static int copy_pageable_h2d(mkp_ctx* ctx, uint8_t* dst, HostSrc hs, size_t src_off, size_t n, cudaStream_t st) {
    const uint8_t* src = hs.mem ? hs.mem + src_off : nullptr;
    if (n < ((size_t)8 << 20)) {
        if (src) { CK(cudaMemcpyAsync(dst, src, n, cudaMemcpyHostToDevice, st)); return 0; }
        std::vector<uint8_t> tmp(n);
        if (!read_fully(hs.fd, tmp.data(), n, hs.fd_off + src_off)) return fail(ctx, "short read from the BAM file");
        CK(cudaMemcpyAsync(dst, tmp.data(), n, cudaMemcpyHostToDevice, st));      // (pageable source: returns after the bytes are staged)
        return 0;
    }
    if (!ctx->pin_ready) {
        int want = 6;
        if (const char* e = getenv("MKP_H2D_THREADS")) want = std::max(1, std::min((int)mkp_ctx::N_PIN, atoi(e)));
        for (int i = 0; i < want; i++) { CK(cudaMallocHost(&ctx->pin[i], mkp_ctx::PIN_BYTES)); CK(cudaEventCreateWithFlags(&ctx->pin_ev[i], cudaEventDisableTiming)); ctx->n_pin = i + 1; }
        ctx->pin_ready = true;
    }
    const size_t piece = mkp_ctx::PIN_BYTES;
    const size_t n_piece = (n + piece - 1) / piece;
    const int nt = (int)std::min<size_t>((size_t)ctx->n_pin, n_piece);
    std::vector<cudaError_t> errs(nt, cudaSuccess);
    std::atomic<bool> read_failed{false};
    auto work = [&](int t) {
        cudaError_t e = cudaSetDevice(ctx->device);
        for (size_t k = t; k < n_piece && e == cudaSuccess; k += nt) {
            const size_t off = k * piece, len = std::min(piece, n - off);
            e = cudaEventSynchronize(ctx->pin_ev[t]);              // the previous transfer out of this buffer is done
            if (e != cudaSuccess) break;
            if (src) memcpy(ctx->pin[t], src + off, len);
            else if (!read_fully(hs.fd, (uint8_t*)ctx->pin[t], len, hs.fd_off + src_off + off)) { read_failed = true; break; }
            e = cudaMemcpyAsync(dst + off, ctx->pin[t], len, cudaMemcpyHostToDevice, st);
            if (e == cudaSuccess) e = cudaEventRecord(ctx->pin_ev[t], st);
        }
        errs[t] = e;
    };
    std::vector<std::thread> th;
    for (int t = 1; t < nt; t++) th.emplace_back(work, t);
    work(0);
    for (auto& x : th) x.join();
    for (cudaError_t e : errs) if (e != cudaSuccess) return fail(ctx, std::string("host to device copy: ") + cudaGetErrorString(e));
    if (read_failed) return fail(ctx, "short read from the BAM file");
    return 0;
}

static int bam_load_range_impl(mkp_ctx* ctx, HostSrc hs, size_t file_len, const mkp_bgzf_member* members, size_t n_members,
                               uint64_t inflated_len, uint64_t walk_end, const uint64_t* seeds, size_t n_seeds, size_t* n_records, float* ms);

int mkp_bam_load_range(mkp_ctx* ctx, const uint8_t* file, size_t file_len, const mkp_bgzf_member* members, size_t n_members,
                       uint64_t inflated_len, uint64_t walk_end, const uint64_t* seeds, size_t n_seeds, size_t* n_records, float* ms) {
    if (!file) return -1;
    return bam_load_range_impl(ctx, HostSrc{file, -1, 0}, file_len, members, n_members, inflated_len, walk_end, seeds, n_seeds, n_records, ms);
}

int mkp_bam_load_range_fd(mkp_ctx* ctx, int fd, uint64_t file_off, size_t file_len, const mkp_bgzf_member* members, size_t n_members,
                          uint64_t inflated_len, uint64_t walk_end, const uint64_t* seeds, size_t n_seeds, size_t* n_records, float* ms) {
    if (fd < 0) return -1;
    return bam_load_range_impl(ctx, HostSrc{nullptr, fd, file_off}, file_len, members, n_members, inflated_len, walk_end, seeds, n_seeds, n_records, ms);
}

int mkp_bam_load(mkp_ctx* ctx, const uint8_t* file, size_t file_len, const mkp_bgzf_member* members, size_t n_members,
                 uint64_t inflated_len, const uint64_t* seeds, size_t n_seeds, size_t* n_records, float* ms) {
    return mkp_bam_load_range(ctx, file, file_len, members, n_members, inflated_len, inflated_len, seeds, n_seeds, n_records, ms);
}

static int bam_load_range_impl(mkp_ctx* ctx, HostSrc hs, size_t file_len, const mkp_bgzf_member* members, size_t n_members,
                               uint64_t inflated_len, uint64_t walk_end, const uint64_t* seeds, size_t n_seeds, size_t* n_records, float* ms) {
    if (!ctx || !members || !seeds || !n_seeds) return -1;
    if (walk_end > inflated_len) return fail(ctx, "walk_end lies outside the inflated range");
    if (n_members >= (1u << 24)) return fail(ctx, "too many BGZF members for one load");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    CK(ctx->d_file.ensure(file_len + 64));
    CK(ctx->d_members.ensure(std::max<size_t>(1, n_members) * sizeof(mkp_bgzf_member)));
    CK(ctx->d_bam.ensure(inflated_len + 64));
    CK(ctx->d_seeds.ensure(n_seeds * 8));
    CK(ctx->d_seg_counts.ensure(n_seeds * 4 + 4));
    CK(ctx->d_seg_base.ensure(n_seeds * 4 + 4));
    CK(ctx->d_small.ensure(SMALL_BYTES));
    const uint32_t n_blk = (uint32_t)((n_seeds + 1023) / 1024);
    CK(ctx->d_block_sums.ensure((size_t)n_blk * 4 + 4));
    uint32_t* u = (uint32_t*)(ctx->d_small.as<uint8_t>() + 34 * 8);    // u+10 status, u+11 work, u+12 record count
    CK(cudaEventRecord(ctx->ev[0], st));
    CK(cudaMemcpyAsync(ctx->d_members.p, members, n_members * sizeof(mkp_bgzf_member), cudaMemcpyHostToDevice, st));
    CK(cudaMemcpyAsync(ctx->d_seeds.p, seeds, n_seeds * 8, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(u + 10, 0, 12, st));
    // decoder tables in shared memory (MKP_INFLATE_SMEM=1) or in an L2-resident global scratch (default): see k_inflate
    static const bool tab_global = !(getenv("MKP_INFLATE_SMEM") && getenv("MKP_INFLATE_SMEM")[0] == '1');
    int warps_sm = 28;
    if (const char* e = getenv("MKP_INFLATE_WARPS")) warps_sm = std::max(1, std::min(32, atoi(e)));
    uint32_t hdr_batch = 4;                 // lanes of a warp that run a deflate block header together (k_inflate)
    if (const char* e = getenv("MKP_INFLATE_HDR_BATCH")) hdr_batch = (uint32_t)std::max(1, std::min(32, atoi(e)));
    const size_t smem = tab_global ? 0 : (size_t)INF_THREADS * INF_STRIDE * 2;
    if (!tab_global && !ctx->inflate_attr_set) {      // per device: the opt-in to > 48 KB of dynamic shared memory
        CK(cudaFuncSetAttribute(k_inflate, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        ctx->inflate_attr_set = true;
    }
    const int per_sm = tab_global ? warps_sm : std::max(1, (int)((227 * 1024) / (smem + 1024)));
    uint16_t* gtab = nullptr;
    if (tab_global) {
        CK(ctx->d_inftab.ensure((size_t)ctx->sm_count * per_sm * INF_THREADS * INF_STRIDE * 2));
        gtab = ctx->d_inftab.as<uint16_t>();
    }
    const size_t resident = (size_t)ctx->sm_count * per_sm * INF_THREADS;      // decoders in flight
    // The file goes over in slabs (copy stream); the members of a slab are inflated (compute stream) while the next slab
    // is on the wire. A slab holds at least one round of resident decoders and 128 MB, so small files are a single slab.
    std::vector<size_t> cut;                     // member index where each slab starts
    {
        const size_t min_members = resident, min_bytes = (size_t)128 << 20;
        size_t i0 = 0;
        while (i0 < n_members) {
            cut.push_back(i0);
            size_t i1 = i0;
            const uint64_t b0 = members[i0].in_off;
            while (i1 < n_members && (i1 - i0 < min_members || members[i1].in_off - b0 < min_bytes)) i1++;
            if (n_members - i1 < min_members / 2) i1 = n_members;           // no tiny tail slab
            i0 = i1;
        }
        cut.push_back(n_members);
    }
    const size_t n_slabs = cut.size() - 1;
    CK(ctx->d_slab_work.ensure(std::max<size_t>(1, n_slabs) * 4));
    CK(cudaMemsetAsync(ctx->d_slab_work.p, 0, std::max<size_t>(1, n_slabs) * 4, st));
    CK(cudaEventRecord(ctx->ev_fork, st));
    CK(cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
    CK(cudaEventRecord(ctx->ev[4], ctx->stream2));
    // members are in file order and do not overlap: bytes before the first payload (BGZF headers) travel with their slab
    for (size_t sl = 0; sl < n_slabs; sl++) {
        const size_t a = sl == 0 ? 0 : (size_t)members[cut[sl]].in_off;
        const size_t b = sl + 1 == n_slabs ? file_len : (size_t)members[cut[sl + 1]].in_off;
        if (int rc = copy_pageable_h2d(ctx, ctx->d_file.as<uint8_t>() + a, hs, a, b - a, ctx->stream2)) return rc;
        CK(cudaEventRecord(ctx->ev_join, ctx->stream2));
        CK(cudaStreamWaitEvent(st, ctx->ev_join, 0));
        const size_t nm = cut[sl + 1] - cut[sl];
        const int grid = (int)std::min<size_t>((nm + INF_THREADS - 1) / INF_THREADS, (size_t)ctx->sm_count * per_sm);
        ctx->launches += 1; k_inflate<<<grid, INF_THREADS, smem, st>>>(ctx->d_file.as<uint8_t>(), ctx->d_members.as<mkp_bgzf_member>() + cut[sl], (uint32_t)nm,
                                                  ctx->d_bam.as<uint8_t>(), u + 10, ctx->d_slab_work.as<uint32_t>() + sl, (uint32_t)cut[sl], gtab, hdr_batch);
    }
    CK(cudaEventRecord(ctx->ev[1], ctx->stream2));
    CK(cudaEventRecord(ctx->ev[2], st));
    const int wg = (int)((n_seeds + 127) / 128);
    ctx->launches += 1; k_walk<0><<<wg, 128, 0, st>>>(ctx->d_bam.as<uint8_t>(), walk_end, ctx->d_seeds.as<uint64_t>(), (uint32_t)n_seeds,
                                  ctx->d_seg_counts.as<uint32_t>(), nullptr, nullptr, u + 10);
    ctx->launches += 1; k_block_sum<<<n_blk, 1024, 0, st>>>(ctx->d_seg_counts.as<uint32_t>(), (uint32_t)n_seeds, ctx->d_block_sums.as<uint32_t>());
    ctx->launches += 1; k_scan_blocks<<<1, 1024, 0, st>>>(ctx->d_block_sums.as<uint32_t>(), n_blk, u + 12);
    ctx->launches += 1; k_value_prefix<<<n_blk, 1024, 0, st>>>(ctx->d_seg_counts.as<uint32_t>(), (uint32_t)n_seeds, ctx->d_block_sums.as<uint32_t>(), ctx->d_seg_base.as<uint32_t>());
    uint32_t h[3] = {0, 0, 0};
    CK(cudaMemcpyAsync(h, u + 10, 12, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    if (h[0]) {
        const uint32_t e = h[0];
        if ((e >> 24) & 0x7f) return fail(ctx, "inflate failed (code " + std::to_string((e >> 24) & 0x7f) + ") in BGZF member " + std::to_string(e & 0xffffffu));
        return fail(ctx, (e & 3u) == 2u ? "record chain does not meet a seed offset (stale or foreign index?)" : "corrupt BAM record in the inflated stream");
    }
    const size_t nrec = h[2];
    CK(ctx->d_recs.ensure(std::max<size_t>(1, nrec) * sizeof(mkp_bam_rec)));
    ctx->launches += 1; k_walk<1><<<wg, 128, 0, st>>>(ctx->d_bam.as<uint8_t>(), walk_end, ctx->d_seeds.as<uint64_t>(), (uint32_t)n_seeds,
                                  ctx->d_seg_counts.as<uint32_t>(), ctx->d_seg_base.as<uint32_t>(), ctx->d_recs.as<mkp_bam_rec>(), u + 10);
    CK(cudaEventRecord(ctx->ev[3], st));
    CK(cudaMemcpyAsync(h, u + 10, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    if (h[0]) return fail(ctx, "corrupt BAM record in the inflated stream");
    ctx->bam_len = inflated_len;
    ctx->n_records = nrec;
    if (n_records) *n_records = nrec;
    if (ms) {
        // [0] copy stream busy, [1] start -> last member inflated (copies and inflate overlap), [2] record walk, [3] total
        cudaEventElapsedTime(&ms[0], ctx->ev[4], ctx->ev[1]);
        cudaEventElapsedTime(&ms[1], ctx->ev[0], ctx->ev[2]);
        cudaEventElapsedTime(&ms[2], ctx->ev[2], ctx->ev[3]);
        cudaEventElapsedTime(&ms[3], ctx->ev[0], ctx->ev[3]);
    }
    return 0;
}

int mkp_bam_records(mkp_ctx* ctx, mkp_bam_rec* out) {
    if (!ctx || !out) return -1;
    CK(cudaSetDevice(ctx->device));
    if (ctx->n_records) CK(cudaMemcpy(out, ctx->d_recs.p, ctx->n_records * sizeof(mkp_bam_rec), cudaMemcpyDeviceToHost));
    return 0;
}

int mkp_bam_inflated(mkp_ctx* ctx, uint64_t off, uint8_t* dst, size_t len) {
    if (!ctx || !dst) return -1;
    if (off + len > ctx->bam_len) return fail(ctx, "range outside the inflated stream");
    CK(cudaSetDevice(ctx->device));
    if (len) CK(cudaMemcpy(dst, ctx->d_bam.as<uint8_t>() + off, len, cudaMemcpyDeviceToHost));
    return 0;
}

int mkp_bam_chunk(mkp_ctx* ctx, uint32_t start, uint32_t end, const uint32_t* rec_ids, uint32_t n, const uint32_t* focus_pos, const uint32_t* focus_neg) {
    if (!ctx || (n && !rec_ids)) return -1;
    if (end <= start) return fail(ctx, "empty chunk range");
    if (!ctx->bam_len) return fail(ctx, "mkp_bam_load was not called");
    CK(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    auto now = [] { return std::chrono::steady_clock::now(); };
    auto since = [&](std::chrono::steady_clock::time_point t) { return std::chrono::duration<double>(now() - t).count(); };
    auto t0 = now();
    ctx->n_reads = n; ctx->cs = start; ctx->ce = end;
    ctx->n_words = (end - start + 31) / 32;
    CK(ctx->d_hdrs.ensure(std::max<size_t>(1, n) * sizeof(mkp_read_hdr)));
    CK(ctx->d_entry_off.ensure(((size_t)n + 1) * 8));
    CK(ctx->d_ids.ensure(std::max<size_t>(1, n) * 4));
    CK(ctx->d_plan.ensure(std::max<size_t>(1, n) * sizeof(SlicePlan)));
    CK(ctx->d_need.ensure(std::max<size_t>(1, n) * 4));
    CK(ctx->d_totals.ensure(4 * 8));
    uint64_t tot[4] = {0, 0, 1, 1};
    ctx->slice_prof[0] += since(t0); t0 = now();
    if (n) {
        for (uint32_t i = 0; i < n; i++) if (rec_ids[i] >= ctx->n_records) return fail(ctx, "record id out of range");
        CK(cudaMemcpyAsync(ctx->d_ids.p, rec_ids, (size_t)n * 4, cudaMemcpyHostToDevice, st));
        ctx->launches += 1; k_slice_plan<<<(n + 7) / 8, 256, 0, st>>>(ctx->d_bam.as<uint8_t>(), ctx->d_recs.as<mkp_bam_rec>(), ctx->d_ids.as<uint32_t>(), n,
                                                     ctx->d_hdrs.as<mkp_read_hdr>(), ctx->d_plan.as<SlicePlan>(), ctx->d_need.as<uint32_t>());
        ctx->launches += 1; k_slice_scan<<<1, 1024, 0, st>>>(ctx->d_hdrs.as<mkp_read_hdr>(), ctx->d_need.as<uint32_t>(), n, ctx->d_entry_off.as<uint64_t>(), ctx->d_totals.as<uint64_t>());
        CK(cudaMemcpyAsync(tot, ctx->d_totals.p, 32, cudaMemcpyDeviceToHost, st));
        CK(cudaStreamSynchronize(st));
        CK(cudaGetLastError());
        ctx->slice_prof[1] += since(t0); t0 = now();
        CK(ctx->d_heap.ensure(tot[0] + 64));
        ctx->slice_prof[2] += since(t0); t0 = now();
        const int grid = std::max(1, std::min(ctx->sm_count * 8, (int)((n + 7) / 8)));
        ctx->launches += 1; k_slice_copy<<<grid, 256, 0, st>>>(ctx->d_bam.as<uint8_t>(), ctx->d_hdrs.as<mkp_read_hdr>(), ctx->d_plan.as<SlicePlan>(), n, ctx->d_heap.as<uint8_t>());
    } else {
        CK(cudaMemsetAsync(ctx->d_entry_off.p, 0, 8, st));
        CK(ctx->d_heap.ensure(64));
    }
    ctx->heap_bytes = tot[0];
    ctx->total_entries = tot[1];
    ctx->max_ncigar = (uint32_t)std::max<uint64_t>(1, tot[2]);
    ctx->max_blocks = (uint32_t)((std::max<uint64_t>(1, tot[3]) + 31) / 32);
    ctx->have_focus = focus_pos && focus_neg;
    if (ctx->have_focus) {
        CK(ctx->d_focus_pos.ensure((size_t)ctx->n_words * 4));
        CK(ctx->d_focus_neg.ensure((size_t)ctx->n_words * 4));
        CK(cudaMemcpyAsync(ctx->d_focus_pos.p, focus_pos, (size_t)ctx->n_words * 4, cudaMemcpyHostToDevice, st));
        CK(cudaMemcpyAsync(ctx->d_focus_neg.p, focus_neg, (size_t)ctx->n_words * 4, cudaMemcpyHostToDevice, st));
    }
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    ctx->slice_prof[3] += since(t0); t0 = now();
    const int rc = finish_upload(ctx);
    ctx->slice_prof[4] += since(t0); ctx->slice_prof[5] += 1;
    return rc;
}

int mkp_bam_tags(mkp_ctx* ctx, const uint32_t* rec_ids, uint32_t n, const char* tags, uint32_t n_tags, uint8_t* out) {
    if (!ctx || (n && !rec_ids) || !tags || !out || n_tags == 0 || n_tags > 4) return -1;
    if (!ctx->bam_len) return fail(ctx, "mkp_bam_load was not called");
    CK(cudaSetDevice(ctx->device));
    if (!n) return 0;
    cudaStream_t st = ctx->stream;
    for (uint32_t i = 0; i < n; i++) if (rec_ids[i] >= ctx->n_records) return fail(ctx, "record id out of range");
    CK(ctx->d_ids.ensure((size_t)n * 4));
    CK(ctx->d_plan.ensure(std::max<size_t>(sizeof(SlicePlan), (size_t)n * n_tags * MKP_TAG_CELL)));       // (scratch shared with the slicer)
    CK(ctx->d_small.ensure(SMALL_BYTES));
    uint32_t* u = (uint32_t*)(ctx->d_small.as<uint8_t>() + 34 * 8);
    uint32_t pk[4] = {0, 0, 0, 0};
    for (uint32_t t = 0; t < n_tags; t++) pk[t] = (uint32_t)(uint8_t)tags[2 * t] | ((uint32_t)(uint8_t)tags[2 * t + 1] << 8);
    CK(cudaMemcpyAsync(ctx->d_ids.p, rec_ids, (size_t)n * 4, cudaMemcpyHostToDevice, st));
    CK(cudaMemsetAsync(u + 14, 0, 4, st));
    ctx->launches += 1;
    k_tag_values<<<(n + 7) / 8, 256, 0, st>>>(ctx->d_bam.as<uint8_t>(), ctx->d_recs.as<mkp_bam_rec>(), ctx->d_ids.as<uint32_t>(), n,
                                                 pk[0] | (pk[1] << 16), pk[2] | (pk[3] << 16), n_tags, ctx->d_plan.as<uint8_t>(), u + 14);
    uint32_t ovf = 0;
    CK(cudaMemcpyAsync(out, ctx->d_plan.p, (size_t)n * n_tags * MKP_TAG_CELL, cudaMemcpyDeviceToHost, st));
    CK(cudaMemcpyAsync(&ovf, u + 14, 4, cudaMemcpyDeviceToHost, st));
    CK(cudaStreamSynchronize(st));
    CK(cudaGetLastError());
    if (ovf) return fail(ctx, "a partition tag value is longer than 253 bytes: use --host-ingest for this file");
    return 0;
}

int mkp_fetch_chunk(mkp_ctx* ctx, mkp_read_hdr* hdrs, uint32_t* n_reads, uint8_t* heap, uint64_t* heap_bytes) {
    if (!ctx) return -1;
    CK(cudaSetDevice(ctx->device));
    if (n_reads) *n_reads = ctx->n_reads;
    if (hdrs && ctx->n_reads) CK(cudaMemcpy(hdrs, ctx->d_hdrs.p, (size_t)ctx->n_reads * sizeof(mkp_read_hdr), cudaMemcpyDeviceToHost));
    if (heap && heap_bytes) {
        if (*heap_bytes < ctx->heap_bytes) return fail(ctx, "heap buffer too small");
        if (ctx->heap_bytes) CK(cudaMemcpy(heap, ctx->d_heap.p, ctx->heap_bytes, cudaMemcpyDeviceToHost));
    }
    if (heap_bytes) *heap_bytes = ctx->heap_bytes;
    return 0;
}

uint64_t mkp_kernel_launches(const mkp_ctx* ctx) { return ctx ? ctx->launches : 0; }

size_t mkp_algorithmic_bytes(const mkp_chunk* ch, size_t n_rows) {
    size_t b = 0;
    for (uint32_t i = 0; i < ch->n_reads; i++) {
        const mkp_read_hdr& h = ch->hdrs[i];
        b += 32 + 4ull * h.n_cigar + (h.l_seq + 1) / 2 + h.len_mm + h.len_ml;
    }
    return b + 40 * n_rows;
}

}  // extern "C"
