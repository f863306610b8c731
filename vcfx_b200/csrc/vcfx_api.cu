// vcfx_api.cu — the C ABI of libvcfx_cuda (include/vcfx_cuda.h): context, pinned
// multi-slot streaming pipeline (H2D || kernels || D2H), and the device-resident entry point.
// No CPU fallback lives here: without a CUDA device every call fails with VCFX_E_NO_DEVICE.
#include "vcfx_cuda.h"
#include "vcfx_kernels.cuh"

#include <algorithm>
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <sched.h>
#include <cstring>
#include <new>
#include <string>
#include <vector>

using namespace vcfx;

static_assert(sizeof(vcfx_ds_row) == 16, "ds_matrix_kernel writes a row's metadata as one 16-byte store");
static_assert((VCFX_F_DS_MATRIX & VCFX_F_DS_BED) == 0, "the two dosage row layouts are separate bits");

// kernel launches go through one macro so that the test-only warp emulator (tests/emu/) can build this file with g++
#ifndef VCFX_LAUNCH
#define VCFX_LAUNCH(kern, grid, block, smem, stream, arg) (kern)<<<(grid), (block), (smem), (stream)>>>(arg)
#endif

namespace {

constexpr size_t DEFAULT_CHUNK = 64u << 20;
constexpr uint32_t EVENT_CAP = 1u << 20;
constexpr int MAX_SLOTS = 8;

typedef void (*kernel_fn)(const KParams);

// What the host side needs to know about an operation, one row per vcfx_op (create() sets up the rest: allele_counter's
// selection, genotype_query's query, inbreeding_calculator's per-sample state, the dosage matrix)
struct OpInfo {
    kernel_fn scan;
    kernel_fn general;      // finishes the tiles the lattice kernel left (tile-resume array), or null
    kernel_fn format;       // writes the rows from the row records, or null (no records)
    bool copy;              // the output is the input with lines dropped or rewritten (md_copy_kernel): tail arrays, 8 CTAs per SM
    bool raw_events;        // events are (offset << 2 | reason) words of dropped lines, and every one is kept (the list grows)
    bool row_prefix;        // rows keep a 32-byte copy of their prefix
    bool codes;             // the scan leaves a genotype code per sample column, one byte per input byte
    bool reruns;            // a chunk may have to run again (more rows or text than sized for); a shared chunk is then copied
    size_t (*out_bytes)(unsigned flags, size_t chunk);   // default output slot for chunks of `chunk` bytes
};

static_assert(VCFX_OP_VARIANT_COUNT == OP_VC && VCFX_OP_ALLELE_FREQ == OP_AF && VCFX_OP_HWE == OP_HWE && VCFX_OP_MISSING_DETECT == OP_MD &&
              VCFX_OP_ALLELE_COUNT == OP_AC && VCFX_OP_NONREF_FILTER == OP_NR && VCFX_OP_INDEX == OP_IX && VCFX_OP_PHASE_CHECK == OP_PC &&
              VCFX_OP_INBREEDING == OP_IB && VCFX_OP_GENOTYPE_QUERY == OP_GQ && VCFX_OP_DOSAGE == OP_DS, "OPS is indexed by vcfx_op");
constexpr OpInfo OPS[] = {
    //  scan                        general                     format                       copy   raw    prefix codes  reruns
    {vcfx_scan_kernel<OP_VC, 0>,  nullptr,                    nullptr,                     false, false, false, false, false,
     [](unsigned, size_t) -> size_t { return 4096; }},
    {vcfx_scan_kernel<OP_AF, 0>,  vcfx_scan_kernel<OP_AF, 1>,  format_rows_kernel<OP_AF>,   false, false, true,  false, true,
     [](unsigned, size_t c) -> size_t { return c / 4 + (1u << 20); }},          // rows are ~0.3 % of the input
    {vcfx_scan_kernel<OP_HWE, 0>, vcfx_scan_kernel<OP_HWE, 1>, format_rows_kernel<OP_HWE>,  false, false, true,  false, true,
     [](unsigned, size_t c) -> size_t { return c / 4 + (1u << 20); }},
    {vcfx_scan_kernel<OP_MD, 0>,  nullptr,                    md_copy_kernel,              true,  false, false, false, true,
     [](unsigned, size_t c) -> size_t { return c + c / 4 + 4096; }},
    {vcfx_scan_kernel<OP_AC, 0>,  nullptr,                    format_rows_kernel<OP_AC>,   false, false, false, false, true,
     [](unsigned flags, size_t c) -> size_t {
         if (flags & VCFX_F_AC_AGGREGATE) return c / 4 + (1u << 20);
         if (flags & VCFX_F_AC_BINARY) return c + 4096;
         return 10 * c + 4096;                                                  // a text row per genotype: ~9x the input at 2,504 samples
     }},
    {vcfx_scan_kernel<OP_NR, 0>,  nullptr,                    md_copy_kernel,              true,  false, false, false, true,
     [](unsigned, size_t c) -> size_t { return c + 4096; }},                    // never longer than the input plus one '\n'
    {vcfx_scan_kernel<OP_IX, 0>,  nullptr,                    format_rows_kernel<OP_IX>,   false, false, false, false, true,
     [](unsigned, size_t c) -> size_t { return c / 4 + (1u << 20); }},
    {vcfx_scan_kernel<OP_PC, 0>,  nullptr,                    md_copy_kernel,              true,  true,  false, false, true,
     [](unsigned, size_t c) -> size_t { return c + 4096; }},
    {vcfx_scan_kernel<OP_IB, 0>,  nullptr,                    ib_rows_kernel,              false, false, false, true,  true,
     [](unsigned, size_t) -> size_t { return 1u << 20; }},                      // create() sizes it from the names
    {vcfx_scan_kernel<OP_GQ, 0>,  nullptr,                    md_copy_kernel,              true,  true,  false, false, true,
     [](unsigned, size_t c) -> size_t { return c + 4096; }},
    // text: a sample column of two bytes or more gives at most two.  Matrix: a row takes 16 + W bytes, no more than its line
    // when the line has W columns of two bytes or more (W >= 7); .bed: 16 + ceil(W / 4), less still; rows of fewer columns
    // grow the slot once
    {vcfx_scan_kernel<OP_DS, 0>,  nullptr,                    ds_rows_kernel,              false, false, false, true,  true,
     [](unsigned, size_t c) -> size_t { return c + 4096; }},
};
constexpr int N_OPS = (int)(sizeof OPS / sizeof OPS[0]);

struct Work {                      // device-side bookkeeping for one launch
    uint32_t *tile_lines = nullptr;
    unsigned long long *tile_out = nullptr;
    unsigned long long *tile_base = nullptr;
    unsigned long long *line_base = nullptr;
    uint32_t *tail_start = nullptr, *tail_len = nullptr, *tail_off = nullptr;   // MISSING_DETECT
    uint2 *col_scratch = nullptr;   // ALLELE_COUNT
    unsigned int *ticket = nullptr;      // two counters: [0] lattice / only kernel, [1] general kernel
    uint32_t *tile_resume = nullptr;
    Rec *recs = nullptr;
    uint8_t *rec_prefix = nullptr;
    uint64_t rec_cap = 0;
    DevStats *d_stats = nullptr;
    unsigned long long *events = nullptr;
    uint32_t ev_cap = 0;                 // entries in events (phase_checker grows it when a chunk drops more lines)
    // inbreeding_calculator: a code per sample column (as many bytes as the chunk), the rows in file order, the chunk's place in the order
    uint8_t *ib_codes = nullptr; size_t ib_codes_cap = 0;
    IbMeta *ib_rows = nullptr; uint64_t ib_rows_cap = 0;
    uint8_t *ib_panels = nullptr; uint64_t ib_panel_cap = 0;
    unsigned long long ib_seq = 0; bool ib_first = false;
    DevStats *h_stats = nullptr;   // pinned: results of the last launch
    DevStats *h_init = nullptr;    // pinned: constant initial value uploaded before every launch
    uint32_t tiles_cap = 0;
    cudaEvent_t ev_k0 = nullptr, ev_k1 = nullptr;
    cudaEvent_t ev_stats = nullptr;     // the launch's DevStats have landed in h_stats
};

struct Slot {
    char *h_in = nullptr;          // pinned
    uint8_t *d_in = nullptr;
    uint8_t *d_out = nullptr;
    char *h_out = nullptr;         // pinned
    cudaStream_t stream = nullptr;
    Work w;
    size_t nbytes = 0;
    size_t out_cap = 0;
    vcfx_chunk_info info = {0, 1, 0, 0};
    bool in_flight = false;
    cudaEvent_t ev_h2d = nullptr;          // the chunk is on the device (H2D + pad done)
    cudaEvent_t ev_shared_done = nullptr;  // a secondary context finished reading this slot's d_in
    bool shared_pending = false;
    uint8_t *d_in_used = nullptr;          // the device input of the chunk in flight (own d_in, or a primary's)
    bool d2h_issued = false;               // the text of the chunk in flight is already on its way to h_out
    size_t d2h_bytes = 0;
};

}  // namespace

struct vcfx_ctx {
    vcfx_cfg cfg;
    const OpInfo *op = nullptr;          // OPS[cfg.op]
    kernel_fn format = nullptr;          // the row writer launched behind the scan (op->format, or allele_counter's / the matrix's)
    bool two_pass = false;               // allele_counter text / binary: rows are sized in a first scan and written in a second
    bool ds_matrix = false;              // dosage_calculator with VCFX_F_DS_MATRIX or VCFX_F_DS_BED: rows of 16 + ds_row_bytes
    uint64_t ds_row_bytes = 0;           // W (int8 matrix) or ceil(W / 4) (.bed)
    int device = 0;
    int sm_count = 0;
    int blocks_per_sm = 1;
    size_t chunk_bytes = 0, out_bytes = 0;
    uint32_t tile_bytes = 0;
    size_t line_hint = 0;                // typical bytes per data line (0 = unknown): long lines want larger tiles
    bool line_hint_fixed = false;        // set through vcfx_cuda_set_line_hint
    int n_slots = 0;
    Slot slots[MAX_SLOTS];
    int head = 0;                  // next slot to acquire
    int tail = 0;                  // oldest slot in flight
    int n_in_flight = 0;
    int acquired_slot = -1;
    // device-resident path
    Work dev_work;
    cudaStream_t dev_stream = nullptr;
    bool dev_stream_owned = false;
    bool dev_pending = false;
    size_t dev_nbytes = 0;
    uint8_t *dev_in = nullptr, *dev_out = nullptr;
    size_t dev_out_cap = 0;
    vcfx_chunk_info dev_info = {0, 1, 0, 0};
    // allele_counter selection (device copies); max_col = 0 for the other ops (no column scratch)
    uint32_t n_sel = 0, max_col = 0;
    uint32_t *d_sel_col = nullptr, *d_name_off = nullptr;
    uint8_t *d_names = nullptr;
    uint4 *d_names16 = nullptr;          // one zero-padded 16-byte slot per selected name + tab, when they all have the same length
    uint32_t name_len = 0;
    bool ac_bulk = true;                 // staged rows leave shared memory through cp.async.bulk (VCFX_AC_BULK=0: 128-bit stores)
    int ac_fmt = 0;
    bool ac_ident = false;               // allele_counter selection = columns 0 .. n_sel-1 in order
    bool ac_spec = false;                // allele_counter text: rows are sized by speculation until a chunk has a count of two digits
    bool c4_bulk = false;                // VCFX_C4_BULK=1: the skip-ahead loop reads through the bulk-copy ring (see vcfx_kernels.cuh)
    // genotype_query: the query and what parseDiploidAlleles leaves of it
    uint8_t gq_query[64] = {0}; uint32_t gq_len = 0; int gq_a = -1, gq_b = -1;
    // inbreeding_calculator (d_ib is null for the other ops): the per-sample state that lives from chunk to chunk, and the
    // order the chunks are applied in
    IbState *d_ib = nullptr; double *d_ib_sum = nullptr; unsigned long long *d_ib_het = nullptr; unsigned int *d_ib_used = nullptr; uint8_t *d_ib_last = nullptr;
    cudaEvent_t ib_event = nullptr;      // the last chunk launched has been applied
    bool ib_event_set = false;
    unsigned long long ib_next_seq = 0;
    bool ib_open = false;                // a stream is under way (its final chunk has not been submitted yet)
    // last drained chunk's short-line list
    std::vector<uint64_t> last_events;
    uint64_t last_n_events = 0;
    std::string last_error;
};

namespace {

#define CU(call)                                                                         \
    do {                                                                                 \
        cudaError_t _e = (call);                                                         \
        if (_e != cudaSuccess) {                                                         \
            ctx->last_error = std::string(#call) + ": " + cudaGetErrorString(_e);       \
            return (_e == cudaErrorMemoryAllocation) ? VCFX_E_NOMEM : VCFX_E_CUDA;       \
        }                                                                                \
    } while (0)

#ifdef VCFX_EMU
struct HweArgs { const int32_t *c; size_t n; double *p; };
void hwe_pvalue_entry(const HweArgs a) { hwe_pvalue_kernel(a.c, a.n, a.p); }
void hwe_pvalue_launch(int grid, const int32_t *c, size_t n, double *p) { HweArgs a = {c, n, p}; emu_launch(hwe_pvalue_entry, dim3(grid), dim3(256), 0, nullptr, a); }
#else
void hwe_pvalue_launch(int grid, const int32_t *c, size_t n, double *p) { hwe_pvalue_kernel<<<grid, 256>>>(c, n, p); }
#endif

// Bytes of input owned by one warp.  Larger tiles waste less on the overlap at tile borders (the
// owner of a tile reads on to the end of its last line, and the next owner scans the same bytes for
// its first line start); smaller tiles keep every resident warp busy on small chunks.  Aim for about
// four tiles per resident warp, within [32 KiB, 256 KiB]; cfg.tile_bytes pins it.
constexpr uint32_t MIN_TILE = 32u << 10, MAX_TILE = 256u << 10;

uint32_t tile_for(const vcfx_ctx *ctx, size_t nbytes) {
    if (ctx->tile_bytes) return ctx->tile_bytes;
    size_t warps = (size_t)ctx->sm_count * ctx->blocks_per_sm * WARPS_PER_CTA;
    size_t t = nbytes / (warps * 4 + 1);
    t = (t + 511) & ~(size_t)511;
    t = std::min<size_t>(MAX_TILE, std::max<size_t>(MIN_TILE, t));
    // A tile's owner re-reads about one line around each border (the first-line search and the
    // run-on of its last line): with 70 KB lines and 256 KiB tiles that is +60 % DRAM traffic.  When
    // the typical line length is known, tiles hold at least eight lines as long as every resident
    // warp still gets two tiles.
    if (ctx->line_hint) {
        size_t want = std::min<size_t>((ctx->line_hint * 8 + 511) & ~(size_t)511, (size_t)8 << 20);
        size_t room = (nbytes / (warps * 2 + 1)) & ~(size_t)511;
        t = std::max(t, std::min(want, room));
    }
    return (uint32_t)t;
}

// length of the first data line of a host buffer (0 = none found in the first MiB)
size_t measure_line(const char *p, size_t n, size_t from) {
    size_t pos = std::min(from, n), lim = std::min(n, pos + ((size_t)1 << 20));
    for (int tries = 0; pos < lim && tries < 4096; ++tries) {
        const char *nl = static_cast<const char *>(memchr(p + pos, '\n', lim - pos));
        if (!nl) return 0;
        size_t len = (size_t)(nl - (p + pos)) + 1;
        if (p[pos] != '#' && len > 1) return len;
        pos += len;
    }
    return 0;
}

uint32_t tiles_for(const vcfx_ctx *ctx, size_t nbytes, uint32_t tile) {
    (void)ctx;
    return (uint32_t)std::max<size_t>(1, (nbytes + tile - 1) / tile);
}

int grid_for(const vcfx_ctx *ctx, uint32_t n_tiles) {
    int resident = ctx->sm_count * ctx->blocks_per_sm;
    int need = (int)((n_tiles + WARPS_PER_CTA - 1) / WARPS_PER_CTA);
    return std::max(1, std::min(resident, need));
}

// Row records are sized for ordinary VCFs: one row per 256 input bytes (a line with nine fixed
// fields and a handful of samples is longer than that; at 2,504 samples a line is 10 KB).  If a
// chunk ever has more rows the launch reports overflow and is repeated with the exact count (see
// vcfx_cuda_next_output / vcfx_cuda_sync), and the larger arrays are kept.  64 bytes per record
// (record + prefix copy): 17 MB per 64 MiB chunk, 1.1 GB for a 4.3 GB resident chunk.
uint64_t default_rec_cap(size_t nbytes) { return nbytes / 256 + 65536; }

// Slots are reserved REC_BLOCK at a time per warp and a warp leaves at most one block partly used, so
// the count of a re-run can exceed the count of the run before it by that much (the warps draw
// different tiles the second time).
uint64_t rec_slack(const vcfx_ctx *ctx) {
    return (uint64_t)REC_BLOCK * ctx->sm_count * ctx->blocks_per_sm * WARPS_PER_CTA + 1024;
}

void free_work(Work &w) {
    cudaFree(w.tile_lines); cudaFree(w.tile_out); cudaFree(w.tile_base); cudaFree(w.line_base);
    cudaFree(w.rec_prefix); cudaFree(w.ticket); cudaFree(w.recs); cudaFree(w.d_stats); cudaFree(w.events);
    cudaFree(w.tail_start); cudaFree(w.tail_len); cudaFree(w.tail_off); cudaFree(w.col_scratch); cudaFree(w.tile_resume);
    cudaFree(w.ib_codes); cudaFree(w.ib_rows); cudaFree(w.ib_panels);
    if (w.h_stats) cudaFreeHost(w.h_stats);
    if (w.h_init) cudaFreeHost(w.h_init);
    if (w.ev_k0) cudaEventDestroy(w.ev_k0);
    if (w.ev_k1) cudaEventDestroy(w.ev_k1);
    if (w.ev_stats) cudaEventDestroy(w.ev_stats);
    w = Work();
}

int ensure_work(vcfx_ctx *ctx, Work &w, size_t max_bytes, uint64_t min_recs = 0, uint64_t min_panel_bytes = 0) {
    // sized for the smallest tile any launch of up to max_bytes can pick
    uint32_t tiles = tiles_for(ctx, max_bytes, ctx->tile_bytes ? ctx->tile_bytes : MIN_TILE);
    if (!w.d_stats) {
        CU(cudaMalloc(&w.d_stats, sizeof(DevStats)));
        CU(cudaMalloc(&w.ticket, 2 * sizeof(unsigned int)));
        CU(cudaMalloc(&w.events, sizeof(unsigned long long) * EVENT_CAP));
        w.ev_cap = EVENT_CAP;
        CU(cudaMallocHost(&w.h_stats, sizeof(DevStats)));
        CU(cudaMallocHost(&w.h_init, sizeof(DevStats)));
        memset(w.h_init, 0, sizeof(DevStats)); w.h_init->first_short_key = ~0ULL;
        memset(w.h_stats, 0, sizeof(DevStats));
        CU(cudaEventCreate(&w.ev_k0));
        CU(cudaEventCreate(&w.ev_k1));
        CU(cudaEventCreateWithFlags(&w.ev_stats, cudaEventDisableTiming));
    }
    if (tiles > w.tiles_cap) {
        cudaFree(w.tile_lines); cudaFree(w.tile_out); cudaFree(w.tile_base); cudaFree(w.line_base);
        w.tile_lines = nullptr; w.tile_out = nullptr; w.tile_base = w.line_base = nullptr;
        CU(cudaMalloc(&w.tile_lines, sizeof(uint32_t) * tiles));
        CU(cudaMalloc(&w.tile_out, sizeof(unsigned long long) * tiles));
        CU(cudaMalloc(&w.tile_base, sizeof(unsigned long long) * tiles));
        CU(cudaMalloc(&w.line_base, sizeof(unsigned long long) * tiles));
        if (ctx->op->general) {
            cudaFree(w.tile_resume); w.tile_resume = nullptr;
            CU(cudaMalloc(&w.tile_resume, sizeof(uint32_t) * tiles));
        }
        if (ctx->op->copy) {
            cudaFree(w.tail_start); cudaFree(w.tail_len); cudaFree(w.tail_off);
            w.tail_start = w.tail_len = w.tail_off = nullptr;
            CU(cudaMalloc(&w.tail_start, sizeof(uint32_t) * tiles));
            CU(cudaMalloc(&w.tail_len, sizeof(uint32_t) * tiles));
            CU(cudaMalloc(&w.tail_off, sizeof(uint32_t) * tiles));
        }
        w.tiles_cap = tiles;
    }
    uint64_t recs = 0;
    if (ctx->format) recs = std::max<uint64_t>(default_rec_cap(max_bytes), min_recs);
    if (ctx->max_col && !w.col_scratch) {
        size_t n = (size_t)ctx->sm_count * ctx->blocks_per_sm * WARPS_PER_CTA * std::max<uint32_t>(ctx->max_col, 1);
        CU(cudaMalloc(&w.col_scratch, n * sizeof(uint2)));
    }
    if (ctx->op->codes && max_bytes + VCFX_DEVICE_PAD > w.ib_codes_cap) {
        cudaFree(w.ib_codes); w.ib_codes = nullptr; w.ib_codes_cap = 0;
        CU(cudaMalloc(&w.ib_codes, max_bytes + VCFX_DEVICE_PAD));
        w.ib_codes_cap = max_bytes + VCFX_DEVICE_PAD;
    }
    if (ctx->d_ib) {
        // the codes once more in file order, 32 samples to a panel: lines that have all their columns need less than the
        // input has bytes; min_panel_bytes is what a chunk that did not fit asked for
        const uint64_t want_pan = std::max<uint64_t>(max_bytes + (1u << 20), min_panel_bytes);
        if (want_pan > w.ib_panel_cap) {
            cudaFree(w.ib_panels); w.ib_panels = nullptr; w.ib_panel_cap = 0;
            CU(cudaMalloc(&w.ib_panels, want_pan));
            w.ib_panel_cap = want_pan;
        }
        if (std::max<uint64_t>(recs, w.rec_cap) > w.ib_rows_cap) {
            const uint64_t want = std::max<uint64_t>(recs, w.rec_cap);
            cudaFree(w.ib_rows); w.ib_rows = nullptr; w.ib_rows_cap = 0;
            CU(cudaMalloc(&w.ib_rows, want * sizeof(IbMeta)));
            w.ib_rows_cap = want;
        }
    }
    if (recs > w.rec_cap) {
        cudaFree(w.recs); w.recs = nullptr; w.rec_cap = 0;
        cudaFree(w.rec_prefix); w.rec_prefix = nullptr;
        CU(cudaMalloc(&w.recs, recs * sizeof(Rec)));
        if (ctx->op->row_prefix) CU(cudaMalloc(&w.rec_prefix, recs * 32));
        w.rec_cap = recs;
    }
    return VCFX_OK;
}

// bytes of panels that hold every row the last launch reserved a record for
uint64_t ib_panel_need(const vcfx_ctx *ctx, const Work &w) {
    return (uint64_t)w.h_stats->n_recs * 32u * ((ctx->n_sel + 31u) / 32u) + (1u << 20);
}

// inbreeding_calculator: a NEW chunk takes the next place in the order its context applies chunks in (a chunk that is run
// again keeps its place); the first chunk behind a final one starts a new stream
void ib_begin(vcfx_ctx *ctx, Work &w, const vcfx_chunk_info *info) {
    if (!ctx->d_ib) return;
    w.ib_seq = ctx->ib_next_seq++;
    w.ib_first = !ctx->ib_open;
    ctx->ib_open = !(info ? info->is_final != 0 : true);
}

// enqueue the kernels of one chunk on `st`; results land in w.h_stats after the stream drains
int launch_chunk(vcfx_ctx *ctx, Work &w, cudaStream_t st, uint8_t *d_in, size_t nbytes,
                 const vcfx_chunk_info *info, uint8_t *d_out, size_t out_cap, bool write_pad = true) {
    const OpInfo &op = *ctx->op;
    const uint32_t tile = tile_for(ctx, nbytes);
    uint32_t tiles = tiles_for(ctx, nbytes, tile);
    if (write_pad) CU(cudaMemsetAsync(d_in + nbytes, '\n', 64, st));
    CU(cudaMemsetAsync(w.ticket, 0, 2 * sizeof(unsigned int), st));
    if (op.general) CU(cudaMemsetAsync(w.tile_resume, 0xFF, sizeof(uint32_t) * tiles, st));
    CU(cudaMemcpyAsync(w.d_stats, w.h_init, sizeof(DevStats), cudaMemcpyHostToDevice, st));

    KParams P;
    P.in = d_in; P.n = nbytes;
    P.tile_bytes = tile; P.n_tiles = tiles;
    P.mode = ctx->cfg.mode; P.flags = ctx->cfg.flags;
    P.valid_from = info ? info->data_valid_from : 0;
    P.fmt0_until = info ? info->format_cache_from : 0;
    P.file_offset = info ? info->file_offset : 0;
    P.is_final = info ? info->is_final : 1;
    P.out = d_out; P.out_cap = out_cap;
    P.tile_lines = w.tile_lines; P.tile_out = w.tile_out; P.tile_base = w.tile_base; P.line_base = w.line_base;
    P.tail_start = w.tail_start; P.tail_len = w.tail_len; P.tail_off = w.tail_off;
    P.ac_fmt = ctx->ac_fmt; P.ac_ident = ctx->ac_ident ? 1 : 0; P.ac_pass = 0; P.ac_spec = ctx->ac_spec ? 1 : 0; P.n_sel = ctx->n_sel; P.sel_col = ctx->d_sel_col; P.name_off = ctx->d_name_off;
    P.names = ctx->d_names; P.names16 = ctx->d_names16; P.name_len = ctx->name_len; P.ac_bulk = ctx->ac_bulk ? 1 : 0; P.max_col = ctx->max_col; P.col_scratch = w.col_scratch;
    P.ticket = w.ticket; P.ticket2 = w.ticket + 1; P.tile_resume = w.tile_resume; P.recs = w.recs; P.rec_prefix = w.rec_prefix; P.rec_cap = w.rec_cap;
    P.c4_bulk = ctx->c4_bulk ? 1 : 0;
    memcpy(P.gq_query, ctx->gq_query, sizeof P.gq_query); P.gq_len = ctx->gq_len; P.gq_a = ctx->gq_a; P.gq_b = ctx->gq_b; P.gq_strict = (ctx->cfg.flags & VCFX_F_GQ_STRICT) ? 1 : 0;
    P.ib_codes = w.ib_codes; P.ib_rows = w.ib_rows; P.ib_panels = w.ib_panels; P.ib_panel_cap = w.ib_panel_cap; P.ib = ctx->d_ib; P.ib_seq = w.ib_seq; P.ib_first = w.ib_first ? 1 : 0; P.text_cap = out_cap;
    if (ctx->d_ib) P.out_cap = ~0ULL;       // the scan counts rows there, not bytes of text
    P.ds_matrix = ctx->ds_matrix ? 1 : 0;
    P.unit_bytes = P.ds_matrix ? 16u + ctx->ds_row_bytes : 1u;      // matrix / .bed: rows x (16 + R) <= out_cap once the rows are counted
    P.stats = w.d_stats; P.events = w.events; P.ev_cap = w.ev_cap; P.ev_raw = op.raw_events ? 1 : 0;

    CU(cudaEventRecord(w.ev_k0, st));
    if (nbytes > 0) {
        int grid = grid_for(ctx, tiles);
        VCFX_LAUNCH(op.scan, grid, WARPS_PER_CTA * 32, 0, st, P);
        CU(cudaGetLastError());
        if (op.general) {                // finishes the tiles the lattice kernel left; exits at once when there are none
            const int ggrid = std::max(1, std::min(ctx->sm_count * scan_ctas(ctx->cfg.op, 1), (int)((tiles + WARPS_PER_CTA - 1) / WARPS_PER_CTA)));
            VCFX_LAUNCH(op.general, ggrid, WARPS_PER_CTA * 32, 0, st, P);
            CU(cudaGetLastError());
        }
        VCFX_LAUNCH(tile_scan_kernel, 1, 1024, SCAN_SMEM_BYTES, st, P);
        CU(cudaGetLastError());
        if (ctx->format) {
            VCFX_LAUNCH(ctx->format, ctx->sm_count * (op.copy ? 8 : 16), 256, 0, st, P);
            CU(cudaGetLastError());
        } else if (ctx->two_pass) {
            // rows are sized in the first pass and written in a second one at their scanned offsets
            CU(cudaMemsetAsync(w.ticket, 0, 2 * sizeof(unsigned int), st));
            P.ac_pass = 1;
            VCFX_LAUNCH(op.scan, grid, WARPS_PER_CTA * 32, 0, st, P);
            CU(cudaGetLastError());
        }
    }
    if (ctx->d_ib) {
        // the sample-axis pass: chunks are applied one after the other, whatever stream they were scanned on
        if (ctx->ib_event_set) CU(cudaStreamWaitEvent(st, ctx->ib_event, 0));
        VCFX_LAUNCH(ib_accumulate_kernel, (int)((ctx->n_sel + 31) / 32), 32, 0, st, P);   // (an empty chunk still opens or closes a stream)
        CU(cudaGetLastError());
        VCFX_LAUNCH(ib_finish_kernel, 1, 1024, 0, st, P);
        CU(cudaGetLastError());
        CU(cudaEventRecord(ctx->ib_event, st));
        ctx->ib_event_set = true;
    }
    CU(cudaEventRecord(w.ev_k1, st));
    CU(cudaMemcpyAsync(w.h_stats, w.d_stats, sizeof(DevStats), cudaMemcpyDeviceToHost, st));
    CU(cudaEventRecord(w.ev_stats, st));
    return VCFX_OK;
}

void fill_stats(const Work &w, size_t nbytes, vcfx_chunk_stats *s) {
    if (!s) return;
    memset(s, 0, sizeof *s);
    const DevStats &d = *w.h_stats;
    s->bytes_in = nbytes; s->bytes_out = d.bytes_out;
    s->lines = d.lines; s->data_lines = d.data_lines; s->rows = d.rows; s->flagged = d.flagged;
    s->pre_header = d.pre_header; s->short_lines = d.short_lines;
    s->first_short_line = d.first_short_line; s->n_events = d.n_events;
    s->dots_terminated = d.dots_terminated; s->last_unterminated_flagged = d.last_unterminated_flagged;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, w.ev_k0, w.ev_k1) == cudaSuccess) s->kernel_ms = ms;
}

int fetch_events(vcfx_ctx *ctx, const Work &w, cudaStream_t st) {
    uint64_t nev = std::min<uint64_t>(w.h_stats->n_events, w.ev_cap);
    ctx->last_n_events = w.h_stats->n_events;
    ctx->last_events.resize(nev);
    if (nev) {
        CU(cudaMemcpyAsync(ctx->last_events.data(), w.events, nev * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        std::sort(ctx->last_events.begin(), ctx->last_events.end());
    }
    return VCFX_OK;
}

// phase_checker and genotype_query report every dropped line: a chunk that dropped more lines than the list holds gets a
// longer list (and is run again).  Returns 1 when it grew, 0 when nothing was lost, a negative vcfx_err on failure.
int grow_events(vcfx_ctx *ctx, Work &w) {
    if (!ctx->op->raw_events || w.h_stats->n_events <= w.ev_cap) return 0;
    const uint64_t want = w.h_stats->n_events + (w.h_stats->n_events >> 3) + 1024;
    if (want > 0xFFFFFFFFull) return VCFX_E_OUTPUT_TOO_BIG;
    cudaFree(w.events); w.events = nullptr; w.ev_cap = 0;
    CU(cudaMalloc(&w.events, sizeof(unsigned long long) * want));
    w.ev_cap = (uint32_t)want;
    return 1;
}

// The text of finished chunks starts its way to the host as soon as their kernels are done, oldest first, whenever the
// caller is in the library: the device->host copy of chunk k+1 then runs while the caller writes chunk k out.
void kick_ready(vcfx_ctx *ctx) {
    for (int i = 0, k = ctx->tail; i < ctx->n_in_flight; ++i, k = (k + 1) % ctx->n_slots) {
        Slot &s = ctx->slots[k];
        if (!s.in_flight || s.d2h_issued) continue;
        if (cudaEventQuery(s.w.ev_stats) != cudaSuccess) break;          // not finished: nor is anything behind it
        if (s.w.h_stats->overflow) continue;                             // next_output runs it again
        const size_t nout = (size_t)s.w.h_stats->bytes_out;
        if (nout && cudaMemcpyAsync(s.h_out, s.d_out, nout, cudaMemcpyDeviceToHost, s.stream) != cudaSuccess) { cudaGetLastError(); break; }
        s.d2h_issued = true; s.d2h_bytes = nout;
    }
}

}  // namespace

extern "C" {

int vcfx_cuda_abi_version(void) { return VCFX_CUDA_ABI_VERSION; }

int vcfx_cuda_device_count(int *n) {
    int c = 0;
    cudaError_t e = cudaGetDeviceCount(&c);
    if (n) *n = (e == cudaSuccess) ? c : 0;
    return (e == cudaSuccess && c > 0) ? VCFX_OK : VCFX_E_NO_DEVICE;
}

const char *vcfx_cuda_strerror(int err) {
    switch (err) {
    case VCFX_OK: return "ok";
    case VCFX_E_INVALID: return "invalid argument or call order";
    case VCFX_E_NO_DEVICE: return "no usable CUDA device (libvcfx_cuda has no CPU fallback)";
    case VCFX_E_CUDA: return "CUDA call failed";
    case VCFX_E_NOMEM: return "out of memory";
    case VCFX_E_BUSY: return "all pipeline slots in flight";
    case VCFX_E_EMPTY: return "nothing in flight";
    case VCFX_E_OUTPUT_TOO_BIG: return "chunk output exceeds the output slot";
    case VCFX_E_UNSUPPORTED: return "operation not supported";
    default: return "unknown error";
    }
}

const char *vcfx_cuda_last_error(const vcfx_ctx *ctx) { return ctx ? ctx->last_error.c_str() : ""; }

int vcfx_cuda_create(const vcfx_cfg *cfg, vcfx_ctx **out) {
    if (!cfg || !out) return VCFX_E_INVALID;
    *out = nullptr;
    if (cfg->op < 0 || cfg->op >= N_OPS) return VCFX_E_INVALID;
    if (cfg->mode != VCFX_MODE_FILE && cfg->mode != VCFX_MODE_STDIN) return VCFX_E_INVALID;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return VCFX_E_NO_DEVICE;
    if (cfg->device < 0 || cfg->device >= ndev) return VCFX_E_INVALID;
    vcfx_ctx *ctx = new (std::nothrow) vcfx_ctx();
    if (!ctx) return VCFX_E_NOMEM;
    ctx->cfg = *cfg;
    ctx->op = &OPS[cfg->op];
    ctx->format = ctx->op->format;
    ctx->device = cfg->device;
    ctx->chunk_bytes = cfg->chunk_bytes ? cfg->chunk_bytes : DEFAULT_CHUNK;
    ctx->tile_bytes = cfg->tile_bytes > 0 ? std::max<uint32_t>(512, ((uint32_t)cfg->tile_bytes + 511) & ~511u) : 0;   // 0 = per launch
    ctx->out_bytes = cfg->out_bytes ? cfg->out_bytes : ctx->op->out_bytes(cfg->flags, ctx->chunk_bytes);
    ctx->n_slots = cfg->n_slots > 0 ? std::min(cfg->n_slots, MAX_SLOTS) : 3;
    auto fail = [&](int rc) { std::string e = ctx->last_error; vcfx_cuda_destroy(ctx); (void)e; return rc; };
#define CUC(call)                                                                        \
    do {                                                                                 \
        cudaError_t _e = (call);                                                         \
        if (_e != cudaSuccess) {                                                         \
            ctx->last_error = std::string(#call) + ": " + cudaGetErrorString(_e);       \
            return fail(_e == cudaErrorMemoryAllocation ? VCFX_E_NOMEM : VCFX_E_CUDA);   \
        }                                                                                \
    } while (0)
    CUC(cudaSetDevice(ctx->device));
    cudaDeviceProp prop;
    CUC(cudaGetDeviceProperties(&prop, ctx->device));
    ctx->sm_count = prop.multiProcessorCount;
    int bps = 1;
    CUC(cudaFuncSetAttribute(tile_scan_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SCAN_SMEM_BYTES));
    CUC(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&bps, ctx->op->scan, WARPS_PER_CTA * 32, 0));
    // the kernels are tuned at their __launch_bounds__ occupancy (variant_counter measured slower at 6 CTAs than at 5)
    ctx->blocks_per_sm = std::max(1, std::min(bps, scan_ctas(cfg->op, 0)));
    if (cfg->op == VCFX_OP_ALLELE_COUNT) {
        if (cfg->n_sel == 0 || !cfg->sel_col || !cfg->sel_names || !cfg->sel_name_off) return fail(VCFX_E_INVALID);
        ctx->ac_fmt = (cfg->flags & VCFX_F_AC_AGGREGATE) ? AC_AGG : (cfg->flags & VCFX_F_AC_BINARY) ? AC_BIN
                    : (cfg->flags & VCFX_F_AC_FORWARD) ? AC_TEXT_FWD : AC_TEXT_MT;
        if (ctx->ac_fmt != AC_AGG) { ctx->format = nullptr; ctx->two_pass = true; }
        ctx->ac_spec = ctx->ac_fmt == AC_TEXT_MT;
        std::vector<uint32_t> cols(cfg->sel_col, cfg->sel_col + cfg->n_sel);
        if (ctx->ac_fmt != AC_TEXT_MT)                      // forward-only column walk (:1222-1227): running maximum
            for (size_t i = 1; i < cols.size(); ++i) cols[i] = std::max(cols[i], cols[i - 1]);
        ctx->n_sel = cfg->n_sel;
        ctx->ac_ident = true;
        for (uint32_t i = 0; i < cfg->n_sel; ++i) if (cfg->sel_col[i] != i) { ctx->ac_ident = false; break; }
        ctx->max_col = *std::max_element(cols.begin(), cols.end()) + 1;
        const size_t nb = cfg->sel_name_off[cfg->n_sel];
        CUC(cudaMalloc(&ctx->d_sel_col, sizeof(uint32_t) * cfg->n_sel));
        CUC(cudaMalloc(&ctx->d_name_off, sizeof(uint32_t) * (cfg->n_sel + 1)));
        CUC(cudaMalloc(&ctx->d_names, nb + 16));
        CUC(cudaMemcpy(ctx->d_sel_col, cols.data(), sizeof(uint32_t) * cfg->n_sel, cudaMemcpyHostToDevice));
        CUC(cudaMemcpy(ctx->d_name_off, cfg->sel_name_off, sizeof(uint32_t) * (cfg->n_sel + 1), cudaMemcpyHostToDevice));
        CUC(cudaMemcpy(ctx->d_names, cfg->sel_names, nb, cudaMemcpyHostToDevice));
        // the fast row writer needs every name (with its tab) to have the same length, at most 12 bytes
        uint32_t nl = cfg->sel_name_off[1] - cfg->sel_name_off[0];
        for (uint32_t i = 1; i < cfg->n_sel && nl; ++i) if (cfg->sel_name_off[i + 1] - cfg->sel_name_off[i] != nl) nl = 0;
        if (nl >= 1 && nl <= 12 && !getenv("VCFX_AC_SLOW_ROWS")) {
            std::vector<unsigned char> n16((size_t)cfg->n_sel * 16, 0);
            for (uint32_t i = 0; i < cfg->n_sel; ++i) memcpy(&n16[(size_t)i * 16], cfg->sel_names + cfg->sel_name_off[i], nl);
            CUC(cudaMalloc(&ctx->d_names16, n16.size()));
            CUC(cudaMemcpy(ctx->d_names16, n16.data(), n16.size(), cudaMemcpyHostToDevice));
            ctx->name_len = nl;
            const char *be = getenv("VCFX_AC_BULK");          // staged rows leave shared memory through cp.async.bulk (default; 0 = 128-bit stores)
            ctx->ac_bulk = !(be && *be == '0');
        }
    }
    { const char *be = getenv("VCFX_C4_BULK"); ctx->c4_bulk = be && *be == '1'; }
    if (cfg->op == VCFX_OP_GENOTYPE_QUERY) {
        // cfg.sel_names = the -g argument, cfg.n_sel = its length.  VCFX_genotype_query.cpp:246-272 parseDiploidAlleles on it,
        // keeping whatever the parse assigned before it gave up (:640-644 uses the two numbers whether it succeeded or not)
        if (!cfg->sel_names || cfg->n_sel == 0 || cfg->n_sel >= sizeof ctx->gq_query) return fail(VCFX_E_INVALID);
        ctx->gq_len = cfg->n_sel;
        memcpy(ctx->gq_query, cfg->sel_names, cfg->n_sel);
        if (!(cfg->flags & VCFX_F_GQ_STRICT)) {
            const char *g = cfg->sel_names; const size_t n = cfg->n_sel;
            int a1 = -1, a2 = -1;
            size_t sp = 0;
            while (sp < n && g[sp] != '|' && g[sp] != '/') ++sp;
            bool ok = !(sp == n || sp == 0 || sp == n - 1) && !(sp == 1 && g[0] == '.');
            if (ok) {
                a1 = 0;
                for (size_t i = 0; i < sp && ok; ++i) { if (g[i] < '0' || g[i] > '9') ok = false; else a1 = (int)((unsigned)a1 * 10u + (unsigned)(g[i] - '0')); }
            }
            if (ok && !(n - sp - 1 == 1 && g[sp + 1] == '.')) {
                a2 = 0;
                for (size_t i = sp + 1; i < n; ++i) { if (g[i] < '0' || g[i] > '9') break; a2 = (int)((unsigned)a2 * 10u + (unsigned)(g[i] - '0')); }
            }
            if (a1 > a2) std::swap(a1, a2);
            ctx->gq_a = a1; ctx->gq_b = a2;
        }
    }
    if (cfg->op == VCFX_OP_INBREEDING) {
        // the samples of the "#CHROM" line, in column order: names as for allele_counter (each followed by a tab)
        if (cfg->n_sel == 0 || !cfg->sel_names || !cfg->sel_name_off) return fail(VCFX_E_INVALID);
        ctx->n_sel = cfg->n_sel;
        const size_t nb = cfg->sel_name_off[cfg->n_sel];
        CUC(cudaMalloc(&ctx->d_name_off, sizeof(uint32_t) * (cfg->n_sel + 1)));
        CUC(cudaMalloc(&ctx->d_names, nb + 16));
        CUC(cudaMemcpy(ctx->d_name_off, cfg->sel_name_off, sizeof(uint32_t) * (cfg->n_sel + 1), cudaMemcpyHostToDevice));
        CUC(cudaMemcpy(ctx->d_names, cfg->sel_names, nb, cudaMemcpyHostToDevice));
        CUC(cudaMalloc(&ctx->d_ib_sum, sizeof(double) * cfg->n_sel));
        CUC(cudaMalloc(&ctx->d_ib_het, sizeof(unsigned long long) * cfg->n_sel));
        CUC(cudaMalloc(&ctx->d_ib_used, sizeof(unsigned int) * cfg->n_sel));
        CUC(cudaMalloc(&ctx->d_ib_last, cfg->n_sel));
        CUC(cudaMalloc(&ctx->d_ib, sizeof(IbState)));
        IbState st0; st0.seq = 0; st0.variants = 0; st0.sum = ctx->d_ib_sum; st0.het = ctx->d_ib_het; st0.used = ctx->d_ib_used; st0.last = ctx->d_ib_last;
        CUC(cudaMemcpy(ctx->d_ib, &st0, sizeof st0, cudaMemcpyHostToDevice));
        CUC(cudaEventCreateWithFlags(&ctx->ib_event, cudaEventDisableTiming));
        if (!cfg->out_bytes) ctx->out_bytes = nb + (size_t)cfg->n_sel * 48 + 4096;      // "name \t F \n" per sample
    }
    if (cfg->op == VCFX_OP_DOSAGE && (cfg->flags & (VCFX_F_DS_MATRIX | VCFX_F_DS_BED))) {
        const bool bed = (cfg->flags & VCFX_F_DS_BED) != 0;
        if (bed && (cfg->flags & VCFX_F_DS_MATRIX)) return fail(VCFX_E_INVALID);
        ctx->ds_matrix = true;
        ctx->format = bed ? ds_matrix_kernel<true> : ds_matrix_kernel<false>;
        ctx->n_sel = cfg->n_sel;                                    // W, the sample columns of the matrix (0 is valid)
        ctx->ds_row_bytes = bed ? ((uint64_t)cfg->n_sel + 3) / 4 : cfg->n_sel;
    }
    if (cfg->stream) { ctx->dev_stream = (cudaStream_t)cfg->stream; ctx->dev_stream_owned = false; }
    else { CUC(cudaStreamCreateWithFlags(&ctx->dev_stream, cudaStreamNonBlocking)); ctx->dev_stream_owned = true; }
#undef CUC
    *out = ctx;
    return VCFX_OK;
}

void vcfx_cuda_destroy(vcfx_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    for (int i = 0; i < MAX_SLOTS; ++i) {
        Slot &s = ctx->slots[i];
        if (s.stream) { cudaStreamSynchronize(s.stream); }
        if (s.h_in) cudaFreeHost(s.h_in);
        if (s.h_out) cudaFreeHost(s.h_out);
        cudaFree(s.d_in); cudaFree(s.d_out);
        free_work(s.w);
        if (s.ev_h2d) cudaEventDestroy(s.ev_h2d);
        if (s.ev_shared_done) cudaEventDestroy(s.ev_shared_done);
        if (s.stream) cudaStreamDestroy(s.stream);
    }
    if (ctx->dev_stream) cudaStreamSynchronize(ctx->dev_stream);
    free_work(ctx->dev_work);
    if (ctx->dev_stream_owned && ctx->dev_stream) cudaStreamDestroy(ctx->dev_stream);
    cudaFree(ctx->d_sel_col); cudaFree(ctx->d_name_off); cudaFree(ctx->d_names); cudaFree(ctx->d_names16);
    cudaFree(ctx->d_ib); cudaFree(ctx->d_ib_sum); cudaFree(ctx->d_ib_het); cudaFree(ctx->d_ib_used); cudaFree(ctx->d_ib_last);
    if (ctx->ib_event) cudaEventDestroy(ctx->ib_event);
    delete ctx;
}

// Pinned staging memory should live on the NUMA node the GPU hangs off: with several GPUs fed from one node's memory
// the host fabric, not PCIe, limits the copies (round 1: 22.8 GB/s per GPU at 8 GPUs against 54.7 alone).  Linux
// places pages on the node of the thread that first touches them, and cudaMallocHost touches them in the calling
// thread: for the duration of the allocations the thread is bound to the cores sysfs lists as local to the GPU
// (/sys/bus/pci/devices/<id>/local_cpulist).  VCFX_NUMA=0 switches it off; a box without NUMA information is untouched.
class NumaBind {
  public:
    explicit NumaBind(int device) {
#ifndef VCFX_EMU
        const char *e = getenv("VCFX_NUMA");
        if (e && *e == '0') return;
        char bus[32] = {0};
        if (cudaDeviceGetPCIBusId(bus, (int)sizeof bus, device) != cudaSuccess) { cudaGetLastError(); return; }
        for (char *c = bus; *c; ++c) *c = (char)tolower((unsigned char)*c);
        std::string path = std::string("/sys/bus/pci/devices/") + bus + "/local_cpulist";
        FILE *f = fopen(path.c_str(), "r");
        if (!f) return;
        char line[1024] = {0};
        const bool got = fgets(line, sizeof line, f) != nullptr;
        fclose(f);
        if (!got) return;
        cpu_set_t want; CPU_ZERO(&want);
        int n_want = 0;
        for (const char *p = line; *p && *p != '\n';) {
            char *end = nullptr;
            long a = strtol(p, &end, 10);
            if (end == p) break;
            long b = a;
            if (*end == '-') { p = end + 1; b = strtol(p, &end, 10); }
            for (long c = a; c <= b && c < CPU_SETSIZE; ++c) { CPU_SET((int)c, &want); ++n_want; }
            p = (*end == ',') ? end + 1 : end;
        }
        if (sched_getaffinity(0, sizeof old_, &old_) != 0) return;
        cpu_set_t both; CPU_AND(&both, &want, &old_);
        if (CPU_COUNT(&both) == 0 || CPU_COUNT(&both) == CPU_COUNT(&old_)) return;      // nothing local we may use, or nothing to narrow
        if (sched_setaffinity(0, sizeof both, &both) == 0) bound_ = true;
#else
        (void)device;
#endif
    }
    ~NumaBind() {
#ifndef VCFX_EMU
        if (bound_) sched_setaffinity(0, sizeof old_, &old_);
#endif
    }
    bool bound() const { return bound_; }

  private:
    cpu_set_t old_;
    bool bound_ = false;
};

static int ensure_slot(vcfx_ctx *ctx, Slot &s) {
    if (s.h_in) return VCFX_OK;
    CU(cudaSetDevice(ctx->device));
    NumaBind numa(ctx->device);
    CU(cudaStreamCreateWithFlags(&s.stream, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&s.ev_h2d, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&s.ev_shared_done, cudaEventDisableTiming));
    CU(cudaMallocHost(&s.h_in, ctx->chunk_bytes));
    CU(cudaMalloc(&s.d_in, ctx->chunk_bytes + VCFX_DEVICE_PAD));
    CU(cudaMalloc(&s.d_out, ctx->out_bytes));
    CU(cudaMallocHost(&s.h_out, ctx->out_bytes));
    s.out_cap = ctx->out_bytes;
    return ensure_work(ctx, s.w, ctx->chunk_bytes);
}

// What every submit ends with: the chunk in slot s, its bytes at d_in, is launched on the slot's stream and joins the
// pipeline behind the chunks already in flight.
static int start_chunk(vcfx_ctx *ctx, Slot &s, uint8_t *d_in, size_t nbytes, const vcfx_chunk_info *info) {
    s.info = info ? *info : vcfx_chunk_info{0, 1, 0, 0, 0};
    s.d_in_used = d_in;
    ib_begin(ctx, s.w, &s.info);
    int rc = launch_chunk(ctx, s.w, s.stream, d_in, nbytes, &s.info, s.d_out, s.out_cap, false);
    if (rc != VCFX_OK) return rc;
    s.nbytes = nbytes; s.in_flight = true; s.d2h_issued = false;
    ctx->head = (ctx->head + 1) % ctx->n_slots;
    ctx->n_in_flight++;
    return VCFX_OK;
}

// the chunk's bytes go from host memory (the slot's pinned buffer, or the caller's) to the slot's device input, then start
static int upload_and_start(vcfx_ctx *ctx, Slot &s, const void *host, size_t nbytes, const vcfx_chunk_info *info) {
    CU(cudaSetDevice(ctx->device));
    if (s.shared_pending) { CU(cudaStreamWaitEvent(s.stream, s.ev_shared_done, 0)); s.shared_pending = false; }
    if (!ctx->line_hint_fixed) ctx->line_hint = measure_line(static_cast<const char *>(host), nbytes, info ? (size_t)info->data_valid_from : 0);
    if (nbytes) CU(cudaMemcpyAsync(s.d_in, host, nbytes, cudaMemcpyHostToDevice, s.stream));
    CU(cudaMemsetAsync(s.d_in + nbytes, '\n', 64, s.stream));
    CU(cudaEventRecord(s.ev_h2d, s.stream));
    return start_chunk(ctx, s, s.d_in, nbytes, info);
}

// A launch that ran out of room says why in DevStats::overflow, and phase_checker / genotype_query may have dropped more
// lines than the event list holds.  This grows what was short and returns 1 when the chunk is to run again (its input is
// still on the device), 0 when the result stands (an overflow left in it is then an error), a negative vcfx_err on failure.
// `out` is the slot whose output buffer may grow; the device-resident path passes null, since its caller owns that
// buffer, and an OV_OUTPUT is final there.  The row records always get room for the count plus rec_slack: a re-run for
// any reason may reserve that many more.
static int grow_for_rerun(vcfx_ctx *ctx, Work &w, size_t max_bytes, Slot *out) {
    const int grew = grow_events(ctx, w);
    if (grew < 0) return grew;
    const unsigned long long ov = w.h_stats->overflow & (out ? ~0ULL : ~(unsigned long long)OV_OUTPUT);
    if (!ov && !grew) return 0;
    if (ov & OV_AC_SPEC) ctx->ac_spec = false;
    int rc = ensure_work(ctx, w, max_bytes, w.h_stats->n_recs + rec_slack(ctx), (ov & OV_IB_PANELS) ? ib_panel_need(ctx, w) : 0);
    if (rc != VCFX_OK) return rc;
    if (ov & OV_OUTPUT) {
        const size_t want = std::max((size_t)w.h_stats->bytes_out + (1u << 20), out->out_cap + out->out_cap / 4);
        cudaFree(out->d_out); cudaFreeHost(out->h_out); out->d_out = nullptr; out->h_out = nullptr; out->out_cap = 0;
        CU(cudaMalloc(&out->d_out, want));
        CU(cudaMallocHost(&out->h_out, want));
        out->out_cap = want;
    }
    return 1;
}

int vcfx_cuda_acquire_input(vcfx_ctx *ctx, char **buf, size_t *cap) {
    if (!ctx || !buf || !cap) return VCFX_E_INVALID;
    if (ctx->acquired_slot >= 0) {           // re-acquire returns the same buffer
        *buf = ctx->slots[ctx->acquired_slot].h_in; *cap = ctx->chunk_bytes; return VCFX_OK;
    }
    if (ctx->n_in_flight >= ctx->n_slots) return VCFX_E_BUSY;
    Slot &s = ctx->slots[ctx->head];
    int rc = ensure_slot(ctx, s);
    if (rc != VCFX_OK) return rc;
    ctx->acquired_slot = ctx->head;
    *buf = s.h_in; *cap = ctx->chunk_bytes;
    return VCFX_OK;
}

int vcfx_cuda_submit(vcfx_ctx *ctx, size_t nbytes, const vcfx_chunk_info *info) {
    if (!ctx || ctx->acquired_slot < 0 || nbytes > ctx->chunk_bytes) return VCFX_E_INVALID;
    Slot &s = ctx->slots[ctx->acquired_slot];
    int rc = upload_and_start(ctx, s, s.h_in, nbytes, info);
    if (rc != VCFX_OK) return rc;
    ctx->acquired_slot = -1;
    kick_ready(ctx);
    return VCFX_OK;
}

int vcfx_cuda_submit_host(vcfx_ctx *ctx, const void *host, size_t nbytes, const vcfx_chunk_info *info) {
    if (!ctx || (!host && nbytes) || nbytes > ctx->chunk_bytes || ctx->acquired_slot >= 0) return VCFX_E_INVALID;
    if (ctx->n_in_flight >= ctx->n_slots) return VCFX_E_BUSY;
    Slot &s = ctx->slots[ctx->head];
    int rc = ensure_slot(ctx, s);
    if (rc != VCFX_OK) return rc;
    rc = upload_and_start(ctx, s, host, nbytes, info);
    if (rc != VCFX_OK) return rc;
    kick_ready(ctx);
    return VCFX_OK;
}

int vcfx_cuda_set_line_hint(vcfx_ctx *ctx, size_t line_bytes) {
    if (!ctx) return VCFX_E_INVALID;
    ctx->line_hint = line_bytes; ctx->line_hint_fixed = line_bytes != 0;
    return VCFX_OK;
}

int vcfx_cuda_submit_shared(vcfx_ctx *ctx, vcfx_ctx *primary, const vcfx_chunk_info *info) {
    if (!ctx || !primary || ctx == primary || ctx->device != primary->device || ctx->acquired_slot >= 0) return VCFX_E_INVALID;
    if (primary->n_in_flight == 0) return VCFX_E_EMPTY;
    if (ctx->n_in_flight >= ctx->n_slots) return VCFX_E_BUSY;
    Slot &ps = primary->slots[(primary->head + primary->n_slots - 1) % primary->n_slots];   // its newest chunk
    if (!ps.in_flight || ps.nbytes > ctx->chunk_bytes) return VCFX_E_INVALID;
    Slot &s = ctx->slots[ctx->head];
    int rc = ensure_slot(ctx, s);
    if (rc != VCFX_OK) return rc;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamWaitEvent(s.stream, ps.ev_h2d, 0));                 // the bytes are there
    // An operation that may have to run a chunk again (more rows or more text than its slot was sized for) takes a
    // private device copy (a few tens of microseconds): the primary is then free to reuse its buffer at once and a
    // re-run never reads bytes the primary has overwritten.  variant_counter never re-runs and reads the primary's bytes.
    const bool own_copy = ctx->op->reruns;
    if (own_copy) {
        if (ps.nbytes) CU(cudaMemcpyAsync(s.d_in, ps.d_in, ps.nbytes, cudaMemcpyDeviceToDevice, s.stream));
        CU(cudaMemsetAsync(s.d_in + ps.nbytes, '\n', 64, s.stream));
        CU(cudaEventRecord(ps.ev_shared_done, s.stream));
        ps.shared_pending = true;
    }
    rc = start_chunk(ctx, s, own_copy ? s.d_in : ps.d_in, ps.nbytes, info);
    if (rc != VCFX_OK) return rc;
    if (!own_copy) {
        // the primary may not overwrite that device buffer before this context has read it
        CU(cudaEventRecord(ps.ev_shared_done, s.stream));
        ps.shared_pending = true;
    }
    return VCFX_OK;
}

int vcfx_cuda_next_output(vcfx_ctx *ctx, const char **text, size_t *n, vcfx_chunk_stats *stats) {
    if (!ctx || !text || !n) return VCFX_E_INVALID;
    if (ctx->n_in_flight == 0) return VCFX_E_EMPTY;
    Slot &s = ctx->slots[ctx->tail];
    CU(cudaSetDevice(ctx->device));
    kick_ready(ctx);
    CU(cudaStreamSynchronize(s.stream));            // kernels, stats and (when already issued) the text of this chunk
    s.in_flight = false;
    ctx->tail = (ctx->tail + 1) % ctx->n_slots;
    ctx->n_in_flight--;
    // a chunk with more rows / more text than the slot was sized for is run again; the larger buffers are kept
    for (int attempt = 0; attempt < 3; ++attempt) {
        const int again = grow_for_rerun(ctx, s.w, ctx->chunk_bytes, &s);
        if (again < 0) return again;
        if (!again) break;
        int rc = launch_chunk(ctx, s.w, s.stream, s.d_in_used, s.nbytes, &s.info, s.d_out, s.out_cap, false);
        if (rc != VCFX_OK) return rc;
        CU(cudaStreamSynchronize(s.stream));
        s.d2h_issued = false;
    }
    if (s.w.h_stats->overflow) return VCFX_E_OUTPUT_TOO_BIG;
    size_t nout = (size_t)s.w.h_stats->bytes_out;
    if (!s.d2h_issued && nout) {
        CU(cudaMemcpyAsync(s.h_out, s.d_out, nout, cudaMemcpyDeviceToHost, s.stream));
        CU(cudaStreamSynchronize(s.stream));
    }
    s.d2h_issued = false;
    int rc = fetch_events(ctx, s.w, s.stream);
    if (rc != VCFX_OK) return rc;
    fill_stats(s.w, s.nbytes, stats);
    *text = s.h_out; *n = nout;
    kick_ready(ctx);                                // whatever finished meanwhile starts its copy before the caller leaves
    return VCFX_OK;
}

int vcfx_cuda_in_flight(const vcfx_ctx *ctx) { return ctx ? ctx->n_in_flight : 0; }

int vcfx_cuda_short_lines(vcfx_ctx *ctx, uint64_t *line_no, size_t cap, size_t *n) {
    if (!ctx || !n) return VCFX_E_INVALID;
    size_t k = std::min(cap, ctx->last_events.size());
    if (line_no && k) memcpy(line_no, ctx->last_events.data(), k * sizeof(uint64_t));
    *n = k;
    return VCFX_OK;
}

int vcfx_cuda_run_device(vcfx_ctx *ctx, void *d_in, size_t nbytes, const vcfx_chunk_info *info,
                         void *d_out, size_t out_cap) {
    if (!ctx || !d_in || ((uintptr_t)d_in & 15)) return VCFX_E_INVALID;
    if (ctx->ds_matrix && ((uintptr_t)d_out & 15)) return VCFX_E_INVALID;     // the row metadata is written in 16-byte stores
    CU(cudaSetDevice(ctx->device));
    int rc = ensure_work(ctx, ctx->dev_work, nbytes);
    if (rc != VCFX_OK) return rc;
    ctx->dev_info = info ? *info : vcfx_chunk_info{0, 1, 0, 0, 0};
    ctx->dev_in = (uint8_t *)d_in; ctx->dev_out = (uint8_t *)d_out; ctx->dev_out_cap = out_cap;
    ib_begin(ctx, ctx->dev_work, &ctx->dev_info);
    rc = launch_chunk(ctx, ctx->dev_work, ctx->dev_stream, ctx->dev_in, nbytes, &ctx->dev_info, ctx->dev_out, out_cap);
    if (rc != VCFX_OK) return rc;
    ctx->dev_pending = true; ctx->dev_nbytes = nbytes;
    return VCFX_OK;
}

int vcfx_cuda_sync(vcfx_ctx *ctx, vcfx_chunk_stats *stats) {
    if (!ctx) return VCFX_E_INVALID;
    if (!ctx->dev_pending) return VCFX_E_EMPTY;
    CU(cudaSetDevice(ctx->device));
    CU(cudaStreamSynchronize(ctx->dev_stream));
    ctx->dev_pending = false;
    const int again = grow_for_rerun(ctx, ctx->dev_work, ctx->dev_nbytes, nullptr);       // one re-run at most
    if (again < 0) return again;
    if (again) {
        int rc = launch_chunk(ctx, ctx->dev_work, ctx->dev_stream, ctx->dev_in, ctx->dev_nbytes, &ctx->dev_info,
                              ctx->dev_out, ctx->dev_out_cap);
        if (rc != VCFX_OK) return rc;
        CU(cudaStreamSynchronize(ctx->dev_stream));
    }
    int rc = fetch_events(ctx, ctx->dev_work, ctx->dev_stream);
    if (rc != VCFX_OK) return rc;
    fill_stats(ctx->dev_work, ctx->dev_nbytes, stats);
    if (ctx->dev_work.h_stats->overflow) return VCFX_E_OUTPUT_TOO_BIG;
    return VCFX_OK;
}

int vcfx_cuda_hwe_pvalues(int device, const int32_t *counts, size_t n, double *pvalues) {
    if ((!counts || !pvalues) && n) return VCFX_E_INVALID;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return VCFX_E_NO_DEVICE;
    if (device < 0 || device >= ndev) return VCFX_E_INVALID;
    if (n == 0) return VCFX_OK;
    if (cudaSetDevice(device) != cudaSuccess) return VCFX_E_CUDA;
    int32_t *d_c = nullptr; double *d_p = nullptr;
    int rc = VCFX_OK;
    if (cudaMalloc(&d_c, n * 3 * sizeof(int32_t)) != cudaSuccess || cudaMalloc(&d_p, n * sizeof(double)) != cudaSuccess) rc = VCFX_E_NOMEM;
    if (rc == VCFX_OK && cudaMemcpy(d_c, counts, n * 3 * sizeof(int32_t), cudaMemcpyHostToDevice) != cudaSuccess) rc = VCFX_E_CUDA;
    if (rc == VCFX_OK) {
        const int grid = (int)std::min<size_t>((n + 255) / 256, 148 * 8);
        hwe_pvalue_launch(grid, d_c, n, d_p);
        if (cudaGetLastError() != cudaSuccess || cudaMemcpy(pvalues, d_p, n * sizeof(double), cudaMemcpyDeviceToHost) != cudaSuccess) rc = VCFX_E_CUDA;
    }
    cudaFree(d_c); cudaFree(d_p);
    return rc;
}

}  // extern "C"
